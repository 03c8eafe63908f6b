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
#include <string>
#include <vector>

using namespace avsep;

namespace {

std::string g_create_error;

__global__ void op_to_f32_kernel(const __nv_bfloat16* in, float* out, size_t n) {
  size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i < n) out[i] = __bfloat162float(in[i]);
}

// out[b, t, :] = lerp of x[b, i0(t), :], x[b, i1(t), :]   (F.interpolate linear, align_corners=False; model.py:115)
__global__ void interp_rows_kernel(const float* __restrict__ x, float* __restrict__ out, int N, int T, int d,
                                   float scale) {
  const int t = blockIdx.x, b = blockIdx.y;
  const float sp = fmaxf(scale * (static_cast<float>(t) + 0.5f) - 0.5f, 0.0f);
  int i0 = static_cast<int>(sp);
  if (i0 > N - 1) i0 = N - 1;
  const int i1 = min(i0 + 1, N - 1);
  const float w1 = sp - static_cast<float>(i0), w0 = 1.0f - w1;
  const float* r0 = x + (static_cast<size_t>(b) * N + i0) * d;
  const float* r1 = x + (static_cast<size_t>(b) * N + i1) * d;
  float* o = out + (static_cast<size_t>(b) * T + t) * d;
  for (int c = threadIdx.x; c < d; c += blockDim.x) o[c] = w0 * r0[c] + w1 * r1[c];
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

struct GraphKey {
  int B, T, N, Hh, Ww;
  const void *mixed, *frames, *sep, *masks, *ws;
  const int *lens, *frame_lens;   // the kernels read the lengths at run time: their contents are not part of the key
  bool operator==(const GraphKey& o) const {
    return B == o.B && T == o.T && N == o.N && Hh == o.Hh && Ww == o.Ww && mixed == o.mixed && frames == o.frames &&
           sep == o.sep && masks == o.masks && ws == o.ws && lens == o.lens && frame_lens == o.frame_lens;
  }
};
struct GraphEntry {
  GraphKey key;
  cudaGraphExec_t exec = nullptr;
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
  cudaStream_t aux_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  std::vector<GraphEntry> graphs;
  uint64_t graph_clock = 0;
  cudaStream_t cap_stream = nullptr;
  int profile_spin_us = 3000;
  uint8_t* d_weights = nullptr;
  size_t weight_bytes = 0;
  // device views into d_weights
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
  void* own_ws = nullptr;
  size_t own_ws_bytes = 0;
  // host-path staging
  // host-buffer entry point: two independent I/O slots so that consecutive calls can overlap (copy-in of call i+1
  // with the kernels and copy-out of call i); slot 0 serves the synchronous avsep_forward_host
  struct HostSlot {
    float* io[4] = {nullptr, nullptr, nullptr, nullptr};   // mixed, frames, separated, masks (device)
    size_t cap[4] = {0, 0, 0, 0};
    std::vector<cudaEvent_t> ev;                            // 2 per chunk: copy-in done, kernels done
    cudaEvent_t ev_start = nullptr, ev_end = nullptr;       // ev_end: last copy-out done
    cudaEvent_t ev_lane[3] = {nullptr, nullptr, nullptr};   // last kernels of this slot on each compute lane
  } slot[AVSEP_HOST_SLOTS];
  std::vector<void*> shared_owned, shared_mapped;   // avsep_shared_alloc / avsep_shared_open
  float* synth_waves = nullptr;   // scratch of avsep_synth_batch
  size_t synth_cap = 0;
  cudaStream_t hs[3] = {nullptr, nullptr, nullptr};
  int host_chunk = 0;    // utterances per pipeline chunk of the host path; 0 = auto (see host_submit)
  bool pdl = true;       // programmatic dependent launch between consecutive kernels of a stream
  int host_lanes = 0;    // chunks whose kernels may be in flight at once (own stream + workspace each); 0 = auto
  void* host_ws = nullptr;
  size_t host_ws_bytes = 0;
  cudaStream_t host_comp[3] = {nullptr, nullptr, nullptr};
  // debug
  bool debug = false;
  std::map<std::string, std::pair<float*, size_t>> snaps;
  int64_t launches = 0;
  // per-launch profiling (cudaEvent pairs on the launching stream)
  bool profile = false;
  cudaStream_t prof_stream = nullptr;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  std::vector<std::pair<const char*, size_t>> ev_marks;   // label, index of the start event (stop = +1)
  std::map<std::string, std::pair<int64_t, double>> prof;  // label -> (launches, total ms)
};

namespace {

int fail(avsep_handle* h, const std::string& msg) {
  if (h) h->err = msg; else g_create_error = msg;
  return 1;
}

int prof_begin(avsep_handle* h, const char* label) {
  if (h->ev_used + 2 > h->ev_pool.size()) {
    for (int i = 0; i < 64; ++i) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) return 1;
      h->ev_pool.push_back(e);
    }
  }
  h->ev_marks.emplace_back(label, h->ev_used);
  cudaEventRecord(h->ev_pool[h->ev_used], h->prof_stream);
  return 0;
}
void prof_end(avsep_handle* h) {
  cudaEventRecord(h->ev_pool[h->ev_used + 1], h->prof_stream);
  h->ev_used += 2;
}

#define CKL(label, expr)                                                \
  do {                                                                  \
    if (h->profile && prof_begin(h, label)) return fail(h, "profiling: cudaEventCreate failed"); \
    const char* _e = (expr);                                            \
    if (_e != nullptr) return fail(h, std::string(_e) + " [" #expr "]"); \
    if (h->profile) prof_end(h);                                        \
    ++h->launches;                                                      \
  } while (0)
#define CK(expr) CKL("other", expr)

#define CUDA_OK(expr)                                                                           \
  do {                                                                                          \
    cudaError_t _c = (expr);                                                                    \
    if (_c != cudaSuccess) return fail(h, std::string(#expr ": ") + cudaGetErrorString(_c));    \
  } while (0)

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

void drop_graphs(avsep_handle* h) {   // cached graphs hold raw pointers to weights / workspace
  for (auto& g : h->graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  h->graphs.clear();
}

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

int get_workspace(avsep_handle* h, Workspace& w, void* user_ws, size_t user_bytes, int B, int T, int N, int Hh, int Ww) {
  const size_t need = carve_workspace(h, w, nullptr, B, T, N, Hh, Ww);
  uint8_t* base = nullptr;
  if (user_ws != nullptr) {
    if (user_bytes < need) return fail(h, "workspace too small: see avsep_workspace_bytes");
    if ((reinterpret_cast<uintptr_t>(user_ws) & 1023) != 0) return fail(h, "workspace must be 1024-byte aligned");
    base = static_cast<uint8_t*>(user_ws);
  } else {
    if (h->own_ws_bytes < need) {
      drop_graphs(h);
      if (h->own_ws) cudaFree(h->own_ws);
      h->own_ws = nullptr;
      h->own_ws_bytes = 0;
      CUDA_OK(cudaMalloc(&h->own_ws, need));
      h->own_ws_bytes = need;
    }
    base = static_cast<uint8_t*>(h->own_ws);
  }
  carve_workspace(h, w, base, B, T, N, Hh, Ww);
  return 0;
}

// ---- debug snapshots ---------------------------------------------------------------------------
int snapshot(avsep_handle* h, cudaStream_t s, const char* name, const void* ptr, size_t count, bool is_op) {
  if (!h->debug) return 0;
  auto& slot = h->snaps[name];
  if (slot.second < count) {
    if (slot.first) cudaFree(slot.first);
    slot.first = nullptr;
    CUDA_OK(cudaMalloc(&slot.first, count * sizeof(float)));
  }
  slot.second = count;
  if (is_op && h->cfg.precision == AVSEP_PREC_BF16) {
    op_to_f32_kernel<<<static_cast<unsigned>((count + 255) / 256), 256, 0, s>>>(
        static_cast<const __nv_bfloat16*>(ptr), slot.first, count);
  } else {
    CUDA_OK(cudaMemcpyAsync(slot.first, ptr, count * sizeof(float), cudaMemcpyDeviceToDevice, s));
  }
  return 0;
}

// ---- stage helpers -----------------------------------------------------------------------------
const char* run_visual_cnn(avsep_handle* h, cudaStream_t s, const float* frames, int M, int Hh, int Ww, void* pooled,
                           unsigned long long* trace = nullptr, const int* frame_lens = nullptr, int N = 1) {
  if (Hh == 32 && Ww == 32 && h->cfg.precision == AVSEP_PREC_BF16)
    return launch_visual_cnn_tc(s, frames, M, h->cnn, h->cnn_w2_slabs, h->cnn_w3_rows, pooled, h->num_sms, trace,
                                frame_lens, N);
  return launch_visual_cnn(s, h->cfg.precision, frames, M, Hh, Ww, h->cnn, pooled, h->num_sms, frame_lens, N);
}

// out[M, N] = A[M, K] W[N, K]^T: one tap, densely packed operands
GemmProblem dense(const void* A, int M, int K, const void* W, int N) {
  GemmProblem p{};
  p.A = A; p.lda = K; p.rowsA = M; p.M = M; p.W = W; p.ldw = K; p.N = N; p.K = K; p.taps = 1;
  return p;
}

int linear(avsep_handle* h, cudaStream_t s, const char* label, const void* A, int M, int K, const void* W,
           const float* bias, int N, int act, float* out_f32, void* out_op) {
  const GemmProblem p = dense(A, M, K, W, N);
  GemmEpilogue e;
  e.bias = bias; e.act = act;
  // a GELU whose only consumer is a bf16 operand does not need the fp32-grade erf
  if (act == ACT_GELU && h->cfg.precision == AVSEP_PREC_BF16 && out_f32 == nullptr) e.act = ACT_GELU_BF16;
  e.out_f32 = out_f32; e.ld_f32 = N;
  e.out_op = out_op; e.ld_op = N;
  CKL(label, launch_gemm(s, h->cfg.precision, p, e, h->num_sms));
  return 0;
}

// GEMM (epilogue fields of `e` already set: bias/act/pe/rowmap) followed by
//   x_out = value (+ resid);  out_op = LayerNorm_{g,b}(x_out)   (g == null: out_op = cast(x_out))
// Fused into the GEMM epilogue when the row fits one tile (EPI_LN), otherwise GEMM -> y, then the warp-shuffle
// add+LayerNorm kernel.  rows_out = number of output rows; y = scratch [rows_out, N] fp32.
int gemm_resid_ln(avsep_handle* h, cudaStream_t s, const char* label, const GemmProblem& p, GemmEpilogue e,
                  const float* resid, float* x_out, const float* g, const float* b, void* out_op, int rows_out,
                  float* y) {
  const int prec = h->cfg.precision;
  if (gemm_ln_fusable(p.N)) {
    e.kind = EPI_LN;
    e.resid = resid;
    e.out_f32 = x_out; e.ld_f32 = p.N;
    e.ln_gamma = g; e.ln_beta = b;
    e.out_op = out_op; e.ld_op = p.N;
    CKL(label, launch_gemm(s, prec, p, e, h->num_sms));
    return 0;
  }
  e.kind = EPI_STD;
  e.out_op = nullptr;
  if (resid != nullptr) {
    e.out_f32 = y; e.ld_f32 = p.N;
    CKL(label, launch_gemm(s, prec, p, e, h->num_sms));
    CKL("add_layernorm", launch_add_layernorm(s, prec, resid, y, g, b, x_out, out_op, rows_out, p.N));
  } else {
    e.out_f32 = x_out; e.ld_f32 = p.N;
    CKL(label, launch_gemm(s, prec, p, e, h->num_sms));
    CKL("add_layernorm", launch_add_layernorm(s, prec, x_out, nullptr, g, b, nullptr, out_op, rows_out, p.N));
  }
  return 0;
}

int linear_resid_ln(avsep_handle* h, cudaStream_t s, const char* label, const void* A, int M, int K, const void* W,
                    const float* bias, int N, float* x, const float* g, const float* b, void* out_op, float* y) {
  GemmEpilogue e;
  e.bias = bias;
  return gemm_resid_ln(h, s, label, dense(A, M, K, W, N), e, x, x, g, b, out_op, M, y);
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
int run_stack(avsep_handle* h, cudaStream_t s, int which, StackProblem sp) {
  const bool pro = sp.pro_a != nullptr;
  sp.wstream = which == 0 ? (pro ? h->xs_a : h->xs_a_np) : which == 1 ? (pro ? h->xs_v : h->xs_v_np) : h->xs_f;
  sp.n_layers = which == 2 ? h->cfg.num_fusion_layers : h->cfg.num_encoder_layers;
  sp.cross = which == 2;
  if (sp.cross) sp.kv_ld = sp.n_layers * 2 * h->cfg.d_model;
  sp.act = sp.cross ? ACT_GELU : ACT_RELU;
  sp.F = h->cfg.freq_bins; sp.S = h->cfg.num_speakers;
  CKL(which == 0 ? "layer.audio_enc" : which == 1 ? "layer.visual_enc" : sp.masks ? "layer.fusion_decoder" : "layer.fusion",
      launch_xformer_stack(s, sp, h->num_sms));
  return 0;
}

// One fused kernel per feed-forward sub-layer (ffn_fused_sm100.cu) from this many rows on; below it the unfused GEMM
// pair spreads over more CTAs and wins.
constexpr int FFN_FUSED_MIN_ROWS = 2048;

// Feed-forward sub-layer of layer w: x += W2 act(W1 a_op + b1) + b2; a_op = LN_{g,b}(x).  ffn [M, 4d], y [M, d]: scratch.
int ffn_sublayer(avsep_handle* h, cudaStream_t s, const LayerW& w, int act, int M, float* x, void* a_op, void* ffn,
                 float* y, const float* g, const float* b) {
  const int d = h->cfg.d_model;
  if (ffn_fusable(h->cfg.precision, d) && M >= FFN_FUSED_MIN_ROWS) {
    CKL("ffn.fused", launch_ffn_fused(s, a_op, w.w1, w.b1, w.w2, w.b2, act, x, x, g, b, a_op, M, h->num_sms, nullptr));
    return 0;
  }
  if (linear(h, s, "gemm.ffn1", a_op, M, d, w.w1, w.b1, 4 * d, act, nullptr, ffn)) return 1;
  return linear_resid_ln(h, s, "gemm.ffn2", ffn, M, 4 * d, w.w2, w.b2, d, x, g, b, a_op, y);
}

// nn.TransformerEncoderLayer x L (pre-norm, ReLU FFN; model.py:48-52,59; torch transformer.py:946-950).
// In: x (fp32 residual stream), a_op = LN_{layer0.norm1}(x).  Out: x, a_op = LN_{final}(x) (or cast when final_g == null).
// lens: keys per utterance of a variable-length batch, or null.
int encoder_stack(avsep_handle* h, cudaStream_t s, const std::vector<LayerW>& layers, int B, int L, float* x,
                  float* y, void* a_op, void* qkv, void* attn, void* ffn, const float* final_g, const float* final_b,
                  const int* lens = nullptr) {
  const int d = h->cfg.d_model, H = h->cfg.nhead, M = B * L, prec = h->cfg.precision;
  const size_t os = op_size(h);
  for (size_t l = 0; l < layers.size(); ++l) {
    const LayerW& w = layers[l];
    if (linear(h, s, "gemm.qkv", a_op, M, d, w.w_in, w.b_in, 3 * d, ACT_NONE, nullptr, qkv)) return 1;
    AttnProblem ap{};
    ap.q = qkv; ap.ldq = 3 * d;
    ap.k = static_cast<const uint8_t*>(qkv) + static_cast<size_t>(d) * os;
    ap.v = static_cast<const uint8_t*>(qkv) + static_cast<size_t>(2 * d) * os;
    ap.ldkv = 3 * d;
    ap.out = attn; ap.ldo = d;
    ap.B = B; ap.H = H; ap.hd = d / H; ap.Lq = L; ap.Lk = L; ap.lerp_src = 0; ap.tc_mode = h->attn_tc;
    ap.k_lens = lens;
    CKL("attn.self", launch_attention(s, prec, ap));
    if (linear_resid_ln(h, s, "gemm.out_proj", attn, M, d, w.wo, w.bo, d, x, w.n2g, w.n2b, a_op, y)) return 1;
    const bool last = (l + 1 == layers.size());
    if (ffn_sublayer(h, s, w, ACT_RELU, M, x, a_op, ffn, y, last ? final_g : layers[l + 1].n1g,
                     last ? final_b : layers[l + 1].n1b))
      return 1;
  }
  return 0;
}

// AudioEncoder up to (not including) the transformer: Conv1d+ReLU x2, +PE (model.py:56-58), then the first
// layer's LayerNorm: x_a (fp32) and a_op = LN_{layer0.norm1}(x_a).
// pl.stack_a: the stack kernel computes the first LayerNorm itself, so only the fp32 residual rows are written, and with
// pl.pro it runs Conv1d #2 + ReLU + PE too, on h1.
int audio_frontend(avsep_handle* h, cudaStream_t s, Workspace& w, const float* mixed, const Plan& pl) {
  h->prof_stream = s;
  const int d = h->cfg.d_model, F = h->cfg.freq_bins, B = w.B, T = w.T, prec = h->cfg.precision;
  const int Map = B * (T + 2);
  CKL("prep_audio", launch_prep_audio(s, prec, mixed, w.xp, B, F, T, h->Fp, w.lens));
  {
    GemmProblem p{};
    p.A = w.xp; p.lda = h->Fp; p.rowsA = Map; p.M = Map; p.W = h->wc1; p.ldw = 3 * h->Fp; p.N = d; p.K = h->Fp;
    p.taps = 3; p.tap_stride = h->Fp; p.row_shift = -1;
    GemmEpilogue e;
    e.bias = h->bc1; e.act = ACT_RELU; e.rowmap = ROW_PAD2PAD; e.Lp = T + 2;
    e.lens = w.lens;
    e.out_op = w.h1; e.ld_op = d;
    CKL("gemm.conv1d_0", launch_gemm(s, prec, p, e, h->num_sms));
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
      CKL("gemm.conv1d_2", launch_gemm(s, prec, p, e, h->num_sms));
    } else if (gemm_resid_ln(h, s, "gemm.conv1d_2", p, e, nullptr, w.x_a, h->enc_a[0].n1g, h->enc_a[0].n1b, w.a_op,
                             B * T, w.y_a)) {
      return 1;
    }
  }
  return snapshot(h, s, "audio_embed", w.x_a, static_cast<size_t>(B) * T * d, false);
}

// VisualEncoder up to (not including) the transformer: CNN, pool, frame_proj, +PE (model.py:106-110), then the
// first layer's LayerNorm: x_v (fp32) and v_op = LN_{layer0.norm1}(x_v).  pl.stack_v / pl.pro as in audio_frontend.
int visual_frontend(avsep_handle* h, cudaStream_t s, Workspace& w, const float* frames, const Plan& pl) {
  h->prof_stream = s;
  const int d = h->cfg.d_model, B = w.B, N = w.N;
  const int Mv = B * N;
  CKL("visual_cnn", run_visual_cnn(h, s, frames, Mv, w.Hh, w.Ww, w.pooled, nullptr, w.frame_lens, N));
  if (snapshot(h, s, "visual_pool", w.pooled, static_cast<size_t>(Mv) * 128, true)) return 1;
  if (pl.stack_v && pl.pro) return 0;
  const GemmProblem p = dense(w.pooled, Mv, 128, h->wproj, d);
  GemmEpilogue e;
  e.bias = h->bproj; e.pe = h->pe_v; e.pe_period = N;
  if (pl.stack_v) {
    e.out_f32 = w.x_v; e.ld_f32 = d;
    CKL("gemm.frame_proj", launch_gemm(s, h->cfg.precision, p, e, h->num_sms));
  } else if (gemm_resid_ln(h, s, "gemm.frame_proj", p, e, nullptr, w.x_v, h->enc_v[0].n1g, h->enc_v[0].n1b, w.v_op, Mv,
                           w.y_v)) {
    return 1;
  }
  return snapshot(h, s, "visual_embed", w.x_v, static_cast<size_t>(Mv) * d, false);
}

// CrossModalFusion (model.py:145-149,166-173) as one kernel: the visual rows are interpolated to the audio frame rate
// first, exactly where the reference does it (model.py:114-116, before the K/V projection), and the K|V rows of every
// fusion layer come from one GEMM on those T rows (bf16) unless the visual stack kernel has written them (pl.kvp).
// In: x_a (fp32 residual), x_v (fp32 visual encoder output, N rows per utterance).  Out: a_op = fusion.norm(x) in bf16,
// or with pl.dec separated / masks from the SeparationDecoder inside the same kernel.
int fusion_stack_fused(avsep_handle* h, cudaStream_t s, Workspace& w, const Plan& pl, const float* mixed,
                       float* separated, float* masks) {
  h->prof_stream = s;
  const int d = h->cfg.d_model, B = w.B, T = w.T;
  const int Ma = B * T, Lf = h->cfg.num_fusion_layers;
  if (!pl.kvp) {
    CKL("lerp_kv", launch_lerp_rows(s, w.x_v, d, B, w.N, T, d, w.attn_a, d, w.frame_lens, w.lens));
    if (linear(h, s, "gemm.cross_kv", w.attn_a, Ma, d, h->wkv_all, h->bkv_all, Lf * 2 * d, ACT_NONE, nullptr, w.kvb)) return 1;
  }
  StackProblem sp{};
  sp.x_in = w.x_a; sp.fin_gamma = h->fng; sp.fin_beta = h->fnb; sp.kv = w.kvb;
  sp.B = B; sp.L = T; sp.lens = w.lens;
  if (pl.dec) {
    sp.mixed = mixed; sp.separated = separated; sp.masks = masks;
    return run_stack(h, s, 2, sp);
  }
  sp.out_x = h->debug ? w.x_a : nullptr; sp.out_op = w.a_op;
  if (run_stack(h, s, 2, sp)) return 1;
  return snapshot(h, s, "fused", w.a_op, static_cast<size_t>(Ma) * d, true);
}

// CrossModalFusion, one kernel per layer.  In: x_a residual stream, a_op = LN_{layer0.norm1}(x_a), v_op = visual rows
// (L_src per utterance).  Out: a_op = fusion.norm(x) in operand precision.
int fusion_stack(avsep_handle* h, cudaStream_t s, Workspace& w, int L_src) {
  h->prof_stream = s;
  const int d = h->cfg.d_model, H = h->cfg.nhead, B = w.B, T = w.T, prec = h->cfg.precision;
  const int Ma = B * T, Mv = B * L_src, Lf = h->cfg.num_fusion_layers;
  // K/V projection of every fusion layer in one GEMM on the un-interpolated visual rows
  if (linear(h, s, "gemm.cross_kv", w.v_op, Mv, d, h->wkv_all, h->bkv_all, Lf * 2 * d, ACT_NONE, w.kvn, nullptr)) return 1;
  for (int l = 0; l < Lf; ++l) {
    const LayerW& fw = h->fus[l];
    if (linear(h, s, "gemm.cross_q", w.a_op, Ma, d, fw.w_in, fw.b_in, d, ACT_NONE, nullptr, w.qkv_a)) return 1;
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
        CKL("lerp_kv", launch_lerp_rows(s, w.kvn + static_cast<size_t>(l) * 2 * d, Lf * 2 * d, B, L_src, T, 2 * d, kvi, 2 * d,
                                        w.frame_lens, w.lens));
        ap = tp;
      }
    }
    CKL("attn.cross", launch_attention(s, prec, ap));
    if (linear_resid_ln(h, s, "gemm.out_proj", w.attn_a, Ma, d, fw.wo, fw.bo, d, w.x_a, fw.n2g, fw.n2b, w.a_op, w.y_a))
      return 1;
    const bool last = (l + 1 == Lf);
    if (ffn_sublayer(h, s, fw, ACT_GELU, Ma, w.x_a, w.a_op, w.ffn_a, w.y_a, last ? h->fng : h->fus[l + 1].n1g,
                     last ? h->fnb : h->fus[l + 1].n1b))
      return 1;
  }
  return snapshot(h, s, "fused", w.a_op, static_cast<size_t>(Ma) * d, true);
}

// SeparationDecoder.forward + .separate (model.py:201-220): a_op = fused rows in operand precision.
int decoder_stage(avsep_handle* h, cudaStream_t s, Workspace& w, const float* mixed, float* separated, float* masks) {
  h->prof_stream = s;
  const int d = h->cfg.d_model, F = h->cfg.freq_bins, S = h->cfg.num_speakers, B = w.B, T = w.T;
  const int Ma = B * T;
  if (linear(h, s, "gemm.dec0", w.a_op, Ma, d, h->wdec0, h->bdec0, 2 * d, ACT_GELU, nullptr, w.ffn_a)) return 1;
  GemmEpilogue e;
  e.kind = EPI_TAIL;
  e.bias = h->bdec3;
  e.mixed = mixed; e.masks = masks; e.separated = separated; e.F = F; e.S = S; e.T = T;
  e.lens = w.lens;
  CKL("gemm.dec3_tail", launch_gemm(s, h->cfg.precision, dense(w.ffn_a, Ma, 2 * d, h->wdec3, S * F), e, h->num_sms));
  return 0;
}

int forward_device(avsep_handle* h, cudaStream_t s, Workspace& w, const float* mixed, const float* frames,
                   float* separated, float* masks) {
  const int d = h->cfg.d_model;
  const int Ma = w.B * w.T, Mv = w.B * w.N;
  const Plan pl = forward_plan(h, w.T, w.N);
  h->prof_stream = s;
  if (h->profile && h->profile_spin_us > 0) spin_kernel<<<1, 1, 0, s>>>(1000ull * h->profile_spin_us);
  // The audio and visual branches are independent until the fusion.
  cudaStream_t sv = s;
  if (pl.fork) {
    if (h->aux_stream == nullptr) {
      CUDA_OK(cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
      CUDA_OK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
      CUDA_OK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    }
    sv = h->aux_stream;
    CUDA_OK(cudaEventRecord(h->ev_fork, s));
    CUDA_OK(cudaStreamWaitEvent(sv, h->ev_fork, 0));
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
  if (snapshot(h, sv, "visual_enc", w.x_v, static_cast<size_t>(Mv) * d, false)) return 1;
  // --- audio branch ---
  if (audio_frontend(h, s, w, mixed, pl)) return 1;
  if (pl.stack_a) {
    StackProblem sp{};
    sp.x_in = w.x_a; sp.out_x = w.x_a; sp.out_op = pl.stack_f ? nullptr : w.a_op;
    sp.fin_gamma = h->fus[0].n1g; sp.fin_beta = h->fus[0].n1b;
    sp.B = w.B; sp.L = w.T; sp.lens = w.lens;
    if (pl.pro) {
      sp.pro_a = w.h1; sp.pro_relu = 1; sp.pro_taps = 3; sp.pro_k = d; sp.pro_pitch = w.T + 2;
      sp.pro_rows = w.B * (w.T + 2); sp.pe = h->pe_a;
    }
    if (run_stack(h, s, 0, sp)) return 1;
  } else if (encoder_stack(h, s, h->enc_a, w.B, w.T, w.x_a, w.y_a, w.a_op, w.qkv_a, w.attn_a, w.ffn_a, h->fus[0].n1g,
                           h->fus[0].n1b, w.lens)) {
    return 1;
  }
  if (snapshot(h, s, "audio_enc", w.x_a, static_cast<size_t>(Ma) * d, false)) return 1;
  if (pl.fork) {
    CUDA_OK(cudaEventRecord(h->ev_join, sv));
    CUDA_OK(cudaStreamWaitEvent(s, h->ev_join, 0));
  }
  // --- fusion + decoder ---
  if (pl.stack_f ? fusion_stack_fused(h, s, w, pl, mixed, separated, masks) : fusion_stack(h, s, w, w.N)) return 1;
  return pl.dec ? 0 : decoder_stage(h, s, w, mixed, separated, masks);
}

// Eager on the first use of a (shape, buffer set); captured into a CUDA graph on the second; replayed afterwards.
// The graph bakes in the kernel parameters (tensor maps included), so a replay costs one host call.
int forward_cached(avsep_handle* h, cudaStream_t s, Workspace& w, const void* ws_base, const float* mixed,
                   const float* frames, float* separated, float* masks) {
  if (!h->use_graph || h->profile || h->debug) return forward_device(h, s, w, mixed, frames, separated, masks);
  const GraphKey key{w.B, w.T, w.N, w.Hh, w.Ww, mixed, frames, separated, masks, ws_base, w.lens, w.frame_lens};
  GraphEntry* ent = nullptr;
  for (auto& g : h->graphs)
    if (g.key == key) { ent = &g; break; }
  if (ent == nullptr) {
    if (h->graphs.size() >= 64) {          // evict the least recently used entry
      size_t victim = 0;
      for (size_t i = 1; i < h->graphs.size(); ++i)
        if (h->graphs[i].last_use < h->graphs[victim].last_use) victim = i;
      if (h->graphs[victim].exec) cudaGraphExecDestroy(h->graphs[victim].exec);
      h->graphs.erase(h->graphs.begin() + victim);
    }
    GraphEntry g;
    g.key = key;
    g.last_use = ++h->graph_clock;
    h->graphs.push_back(g);
    return forward_device(h, s, w, mixed, frames, separated, masks);   // warm-up, also sets kernel attributes
  }
  ent->last_use = ++h->graph_clock;
  if (ent->exec == nullptr) {
    if (h->cap_stream == nullptr) CUDA_OK(cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
    CUDA_OK(cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeRelaxed));
    const int rc = forward_device(h, h->cap_stream, w, mixed, frames, separated, masks);
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(h->cap_stream, &graph);
    if (rc != 0) {
      if (graph) cudaGraphDestroy(graph);
      return 1;
    }
    if (ce != cudaSuccess) return fail(h, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce));
    const cudaError_t ci = cudaGraphInstantiate(&ent->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ci != cudaSuccess) {
      ent->exec = nullptr;
      return fail(h, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ci));
    }
    ent->launches = h->launches;
  }
  h->launches = ent->launches;
  CUDA_OK(cudaGraphLaunch(ent->exec, s));
  return 0;
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
  if (cudaSetDevice(cfg->device) != cudaSuccess) return fail(nullptr, "avsep_create: cudaSetDevice failed");
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
  cudaSetDevice(h->cfg.device);
  if (h->d_weights) cudaFree(h->d_weights);
  if (h->own_ws) cudaFree(h->own_ws);
  for (auto& sl : h->slot) {
    for (float* ptr : sl.io)
      if (ptr) cudaFree(ptr);
    for (cudaEvent_t e : sl.ev) cudaEventDestroy(e);
    if (sl.ev_start) cudaEventDestroy(sl.ev_start);
    if (sl.ev_end) cudaEventDestroy(sl.ev_end);
    for (cudaEvent_t e : sl.ev_lane)
      if (e) cudaEventDestroy(e);
  }
  for (void* ptr : h->shared_mapped) cudaIpcCloseMemHandle(ptr);
  for (void* ptr : h->shared_owned) cudaFree(ptr);
  if (h->synth_waves) cudaFree(h->synth_waves);
  if (h->host_ws) cudaFree(h->host_ws);
  for (auto& kv : h->snaps)
    if (kv.second.first) cudaFree(kv.second.first);
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  for (auto& g : h->graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
  if (h->aux_stream) cudaStreamDestroy(h->aux_stream);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  for (int i = 0; i < 3; ++i) {
    if (h->hs[i]) cudaStreamDestroy(h->hs[i]);
    if (h->host_comp[i]) cudaStreamDestroy(h->host_comp[i]);
  }
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
  if (!h) return 1;
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  CUDA_OK(cudaSetDevice(h->cfg.device));
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
  if (h->d_weights) cudaFree(h->d_weights);
  h->d_weights = nullptr;
  CUDA_OK(cudaMalloc(&h->d_weights, ar.bytes.size()));
  h->weight_bytes = ar.bytes.size();
  CUDA_OK(cudaMemcpyAsync(h->d_weights, ar.bytes.data(), ar.bytes.size(), cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaStreamSynchronize(s));
  ar.patch(h->d_weights);
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
  if (!h) return 1;
  if (!mixed_spec || !lip_frames || !separated || !masks) return fail(h, "avsep_forward: null buffer");
  if (check_shape(h, B, T, N, Hh, Ww)) return 1;
  CUDA_OK(cudaSetDevice(h->cfg.device));
  Workspace w;
  if (get_workspace(h, w, workspace, workspace_bytes, B, T, N, Hh, Ww)) return 1;
  w.lens = lengths; w.frame_lens = frame_lengths;
  h->launches = 0;
  return forward_cached(h, static_cast<cudaStream_t>(cuda_stream), w, workspace ? workspace : h->own_ws, mixed_spec,
                        lip_frames, separated, masks);
}

namespace {
int host_submit(avsep_handle* h, const float* mixed_spec, const float* lip_frames, int B, int T, int N, int Hh, int Ww,
                float* separated, float* masks, int slot_id, cudaStream_t s, bool streaming) {
  // Software pipeline over chunks of the batch: H2D of chunk i+1, kernels of chunk i and D2H of chunk i-1 run
  // concurrently on separate streams (PCIe is full duplex), so a call costs ~max(copy-in, compute, copy-out); the
  // two slots extend the same pipeline across consecutive calls.
  if (!mixed_spec || !lip_frames || !separated || !masks) return fail(h, "avsep_forward_host: null buffer");
  if (slot_id < 0 || slot_id >= AVSEP_HOST_SLOTS) return fail(h, "avsep_forward_host_async: slot must be 0 .. AVSEP_HOST_SLOTS - 1");
  if (check_shape(h, B, T, N, Hh, Ww)) return 1;
  CUDA_OK(cudaSetDevice(h->cfg.device));
  avsep_handle::HostSlot& sl = h->slot[slot_id];
  const size_t F = h->cfg.freq_bins, S = h->cfg.num_speakers;
  const size_t mixed_per = F * T, frames_per = static_cast<size_t>(N) * Hh * Ww, out_per = S * F * T;
  const size_t need[4] = {B * mixed_per, B * frames_per, B * out_per, B * out_per};
  for (int i = 0; i < 4; ++i) {
    if (sl.cap[i] < need[i]) {
      if (sl.ev_end) CUDA_OK(cudaEventSynchronize(sl.ev_end));     // the slot's previous call still owns the buffer
      if (sl.io[i]) cudaFree(sl.io[i]);
      sl.io[i] = nullptr;
      sl.cap[i] = 0;
      CUDA_OK(cudaMalloc(&sl.io[i], need[i] * sizeof(float)));
      sl.cap[i] = need[i];
    }
  }
  float *io_mixed = sl.io[0], *io_frames = sl.io[1], *io_sep = sl.io[2], *io_masks = sl.io[3];
  if (h->hs[0] == nullptr) {
    for (int i = 0; i < 3; ++i) CUDA_OK(cudaStreamCreateWithFlags(&h->hs[i], cudaStreamNonBlocking));
  }
  auto make_event = [&](cudaEvent_t& e) -> int {
    if (e == nullptr) CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    return 0;
  };
  if (make_event(sl.ev_start) || make_event(sl.ev_end)) return 1;
  // Chunk size: a stack kernel takes as long for 64 utterances as for 256 (one tile per CTA either way), so chunks are
  // a trade between pipelining inside one call and kernel time.  Measured at B = 256 (tools/e2e_probe.py): the one-call
  // form is fastest with ~56-utterance chunks on two compute lanes (copy-in of chunk i+1 under the kernels of chunk i),
  // the streaming form - where consecutive calls overlap anyway - with 128-utterance chunks on one lane (161 k against
  // 140 k utt-s/s with 64 x 2).
  const int auto_chunk = streaming ? 128 : 56;
  const int want_chunk = h->host_chunk > 0 ? h->host_chunk : auto_chunk;
  const int Bc = want_chunk < B ? want_chunk : B;
  std::vector<int> starts, sizes;
  for (int b0 = 0; b0 < B; b0 += Bc) {
    starts.push_back(b0);
    sizes.push_back((B - b0) < Bc ? (B - b0) : Bc);
  }
  const int nchunks = static_cast<int>(starts.size());
  while (static_cast<int>(sl.ev.size()) < 2 * nchunks) {
    cudaEvent_t e;
    CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    sl.ev.push_back(e);
  }
  // one workspace + compute stream per lane: with small chunks a single forward cannot fill the GPU, so the kernels
  // of consecutive chunks are allowed to overlap
  const int want_lanes = h->host_lanes > 0 ? h->host_lanes : (streaming ? 1 : 2);
  const int lanes = want_lanes > 3 ? 3 : want_lanes;
  Workspace wl[3];
  const size_t per_lane = carve_workspace(h, wl[0], nullptr, Bc, T, N, Hh, Ww);
  if (h->host_ws_bytes < per_lane * lanes) {
    CUDA_OK(cudaDeviceSynchronize());          // the other slot may still be using the old workspace
    drop_graphs(h);
    if (h->host_ws) cudaFree(h->host_ws);
    h->host_ws = nullptr;
    h->host_ws_bytes = 0;
    CUDA_OK(cudaMalloc(&h->host_ws, per_lane * lanes));
    h->host_ws_bytes = per_lane * lanes;
  }
  for (int l = 0; l < lanes; ++l) {
    carve_workspace(h, wl[l], static_cast<uint8_t*>(h->host_ws) + l * per_lane, Bc, T, N, Hh, Ww);
    if (h->host_comp[l] == nullptr) CUDA_OK(cudaStreamCreateWithFlags(&h->host_comp[l], cudaStreamNonBlocking));
    if (make_event(sl.ev_lane[l])) return 1;
  }
  cudaStream_t s_in = h->hs[0], s_out = h->hs[2];
  // order after whatever the caller queued on its stream, and after this slot's previous use: its kernels have read
  // the input buffers (before they are overwritten) and its copy-out has read the output buffers
  CUDA_OK(cudaEventRecord(sl.ev_start, s));
  CUDA_OK(cudaStreamWaitEvent(s_in, sl.ev_start, 0));
  for (int l = 0; l < 3; ++l)
    if (sl.ev_lane[l]) CUDA_OK(cudaStreamWaitEvent(s_in, sl.ev_lane[l], 0));
  for (int l = 0; l < lanes; ++l) {
    CUDA_OK(cudaStreamWaitEvent(h->host_comp[l], sl.ev_start, 0));
    CUDA_OK(cudaStreamWaitEvent(h->host_comp[l], sl.ev_end, 0));
  }
  CUDA_OK(cudaStreamWaitEvent(s_out, sl.ev_start, 0));
  int64_t launches = 0;
  for (int c = 0; c < nchunks; ++c) {
    const size_t b0 = starts[c];
    const int bc = sizes[c];
    const int lane = c % lanes;
    cudaStream_t s_comp = h->host_comp[lane];
    CUDA_OK(cudaMemcpyAsync(io_mixed + b0 * mixed_per, mixed_spec + b0 * mixed_per, bc * mixed_per * 4,
                            cudaMemcpyHostToDevice, s_in));
    CUDA_OK(cudaMemcpyAsync(io_frames + b0 * frames_per, lip_frames + b0 * frames_per, bc * frames_per * 4,
                            cudaMemcpyHostToDevice, s_in));
    CUDA_OK(cudaEventRecord(sl.ev[2 * c], s_in));
    CUDA_OK(cudaStreamWaitEvent(s_comp, sl.ev[2 * c], 0));
    Workspace wc = wl[lane];
    wc.B = bc;
    if (forward_cached(h, s_comp, wc, static_cast<uint8_t*>(h->host_ws) + lane * per_lane, io_mixed + b0 * mixed_per,
                       io_frames + b0 * frames_per, io_sep + b0 * out_per, io_masks + b0 * out_per))
      return 1;
    launches += h->launches;
    CUDA_OK(cudaEventRecord(sl.ev[2 * c + 1], s_comp));
    CUDA_OK(cudaStreamWaitEvent(s_out, sl.ev[2 * c + 1], 0));
    CUDA_OK(cudaMemcpyAsync(separated + b0 * out_per, io_sep + b0 * out_per, bc * out_per * 4,
                            cudaMemcpyDeviceToHost, s_out));
    CUDA_OK(cudaMemcpyAsync(masks + b0 * out_per, io_masks + b0 * out_per, bc * out_per * 4,
                            cudaMemcpyDeviceToHost, s_out));
  }
  h->launches = launches;
  for (int l = 0; l < lanes; ++l) CUDA_OK(cudaEventRecord(sl.ev_lane[l], h->host_comp[l]));
  // The caller's stream is deliberately NOT made to wait for the results: that would chain call i+1 (which is ordered
  // after the caller's stream) behind call i's copy-out.  Results are consumed on the host after avsep_host_wait.
  CUDA_OK(cudaEventRecord(sl.ev_end, s_out));
  return 0;
}
}  // namespace

int avsep_forward_host(avsep_handle* h, const float* mixed_spec, const float* lip_frames, int32_t B, int32_t T,
                       int32_t N, int32_t Hh, int32_t Ww, float* separated, float* masks, void* cuda_stream) {
  if (!h) return 1;
  if (host_submit(h, mixed_spec, lip_frames, B, T, N, Hh, Ww, separated, masks, 0, static_cast<cudaStream_t>(cuda_stream), false))
    return 1;
  CUDA_OK(cudaEventSynchronize(h->slot[0].ev_end));
  return 0;
}

int avsep_forward_host_async(avsep_handle* h, const float* mixed_spec, const float* lip_frames, int32_t B, int32_t T,
                             int32_t N, int32_t Hh, int32_t Ww, float* separated, float* masks, int32_t slot,
                             void* cuda_stream) {
  if (!h) return 1;
  return host_submit(h, mixed_spec, lip_frames, B, T, N, Hh, Ww, separated, masks, slot,
                     static_cast<cudaStream_t>(cuda_stream), true);
}

int avsep_host_wait(avsep_handle* h, int32_t slot) {
  if (!h) return 1;
  if (slot < 0 || slot >= AVSEP_HOST_SLOTS) return fail(h, "avsep_host_wait: slot must be 0 .. AVSEP_HOST_SLOTS - 1");
  if (h->slot[slot].ev_end == nullptr) return 0;       // nothing was ever submitted on this slot
  CUDA_OK(cudaSetDevice(h->cfg.device));
  CUDA_OK(cudaEventSynchronize(h->slot[slot].ev_end));
  return 0;
}

int avsep_synth_batch(avsep_handle* h, const avsep_synth_config* cfg, int32_t B, const double* amps, const double* freqs,
                      const double* phases, const float* noise, float* mixed_spec, float* lip_frames,
                      float* clean_specs, void* cuda_stream) {
  if (!h) return 1;
  if (!cfg || !amps || !freqs || !phases || !mixed_spec || !lip_frames) return fail(h, "avsep_synth_batch: null argument");
  if (B < 1) return fail(h, "avsep_synth_batch: empty batch");
  CUDA_OK(cudaSetDevice(h->cfg.device));
  SynthProblem p{};
  p.B = B; p.S = cfg->num_speakers; p.n = cfg->num_samples_audio; p.nfft = cfg->n_fft; p.hop = cfg->hop_length;
  p.nf = cfg->num_frames; p.Hh = cfg->frame_h; p.Ww = cfg->frame_w; p.duration = cfg->duration;
  p.amps = amps; p.freqs = freqs; p.phases = phases; p.noise = noise;
  p.mixed_spec = mixed_spec; p.lip_frames = lip_frames; p.clean_specs = clean_specs;
  if (p.S < 1 || p.n < 1) return fail(h, "avsep_synth_batch: bad geometry");
  const size_t need = static_cast<size_t>(B) * (p.S + 1) * p.n;
  if (h->synth_cap < need) {
    if (h->synth_waves) cudaFree(h->synth_waves);
    h->synth_waves = nullptr; h->synth_cap = 0;
    CUDA_OK(cudaMalloc(&h->synth_waves, need * sizeof(float)));
    h->synth_cap = need;
  }
  p.waves = h->synth_waves;
  h->launches = 0;
  CK(launch_synth(static_cast<cudaStream_t>(cuda_stream), p));
  h->launches = 3;
  return 0;
}

int avsep_eval_snr(avsep_handle* h, const float* separated, const float* targets, const float* mixed, int32_t B,
                   int32_t S, int32_t F, int32_t T, double* input_snr, double* output_snr, int32_t* best_perm,
                   double* si_snr, void* cuda_stream) {
  if (!h) return 1;
  if (!separated || !targets) return fail(h, "avsep_eval_snr: null argument");
  if (B < 1 || F < 1 || T < 1) return fail(h, "avsep_eval_snr: empty problem");
  CUDA_OK(cudaSetDevice(h->cfg.device));
  CK(launch_eval_snr(static_cast<cudaStream_t>(cuda_stream), separated, targets, mixed, B, S, F * T, input_snr,
                     output_snr, best_perm, si_snr));
  h->launches = 1;
  return 0;
}

int avsep_stft(avsep_handle* h, const float* waves, int32_t B, int32_t L, int32_t n_fft, int32_t hop_length,
               float* spec, float* mag, void* cuda_stream) {
  return avsep_stft_varlen(h, waves, nullptr, B, L, n_fft, hop_length, spec, mag, nullptr, cuda_stream);
}

int avsep_stft_varlen(avsep_handle* h, const float* waves, const int32_t* lengths, int32_t B, int32_t L, int32_t n_fft,
                      int32_t hop_length, float* spec, float* mag, int32_t* frame_lengths_out, void* cuda_stream) {
  if (!h) return 1;
  if (!waves || !spec) return fail(h, "avsep_stft: null argument");
  CUDA_OK(cudaSetDevice(h->cfg.device));
  CK(launch_stft_complex(static_cast<cudaStream_t>(cuda_stream), waves, lengths, B, L, n_fft, hop_length, spec, mag,
                         frame_lengths_out));
  h->launches = 1;
  return 0;
}

int avsep_istft(avsep_handle* h, const float* spec, const float* masks, int32_t B, int32_t S, int32_t T,
                int32_t n_fft, int32_t hop_length, int32_t L, float* waves, void* cuda_stream) {
  return avsep_istft_varlen(h, spec, masks, nullptr, B, S, T, n_fft, hop_length, L, waves, cuda_stream);
}

int avsep_istft_varlen(avsep_handle* h, const float* spec, const float* masks, const int32_t* lengths, int32_t B,
                       int32_t S, int32_t T, int32_t n_fft, int32_t hop_length, int32_t L, float* waves,
                       void* cuda_stream) {
  if (!h) return 1;
  if (!spec || !waves) return fail(h, "avsep_istft: null argument");
  CUDA_OK(cudaSetDevice(h->cfg.device));
  CK(launch_istft_masked(static_cast<cudaStream_t>(cuda_stream), spec, masks, lengths, B, S, T, n_fft, hop_length, L,
                         waves));
  h->launches = 1;
  return 0;
}

int64_t avsep_last_launch_count(const avsep_handle* h) { return h ? h->launches : 0; }

// ---- batch sharding over the GPUs of one box: peer-mapped buffers + copy-engine transfers (SURVEY 8e) ----------
int avsep_shared_alloc(avsep_handle* h, size_t bytes, void** dev_ptr, unsigned char handle_out[AVSEP_IPC_HANDLE_BYTES]) {
  if (!h) return 1;
  if (!dev_ptr || !handle_out || bytes == 0) return fail(h, "avsep_shared_alloc: bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == AVSEP_IPC_HANDLE_BYTES, "IPC handle size");
  CUDA_OK(cudaSetDevice(h->cfg.device));
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
  for (size_t i = 0; i < h->shared_owned.size(); ++i)
    if (h->shared_owned[i] == dev_ptr) {
      CUDA_OK(cudaSetDevice(h->cfg.device));
      h->shared_owned.erase(h->shared_owned.begin() + i);
      CUDA_OK(cudaFree(dev_ptr));
      return 0;
    }
  return fail(h, "avsep_shared_free: pointer was not allocated by avsep_shared_alloc on this handle");
}

int avsep_shared_open(avsep_handle* h, const unsigned char handle[AVSEP_IPC_HANDLE_BYTES], void** dev_ptr) {
  if (!h) return 1;
  if (!handle || !dev_ptr) return fail(h, "avsep_shared_open: bad argument");
  CUDA_OK(cudaSetDevice(h->cfg.device));
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
  for (size_t i = 0; i < h->shared_mapped.size(); ++i)
    if (h->shared_mapped[i] == dev_ptr) {
      CUDA_OK(cudaSetDevice(h->cfg.device));
      h->shared_mapped.erase(h->shared_mapped.begin() + i);
      CUDA_OK(cudaIpcCloseMemHandle(dev_ptr));
      return 0;
    }
  return fail(h, "avsep_shared_close: pointer was not mapped by avsep_shared_open on this handle");
}

int avsep_copy_async(avsep_handle* h, void* dst, const void* src, size_t bytes, void* cuda_stream) {
  if (!h) return 1;
  if (!dst || !src) return fail(h, "avsep_copy_async: null buffer");
  if (bytes == 0) return 0;
  CUDA_OK(cudaSetDevice(h->cfg.device));
  CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, static_cast<cudaStream_t>(cuda_stream)));
  return 0;
}

int avsep_separate(avsep_handle* h, const float* masks, const float* mixed_spec, int32_t B, int32_t T, float* separated,
                   void* cuda_stream) {
  return avsep_separate_varlen(h, masks, mixed_spec, nullptr, B, T, separated, cuda_stream);
}

int avsep_separate_varlen(avsep_handle* h, const float* masks, const float* mixed_spec, const int32_t* lengths,
                          int32_t B, int32_t T, float* separated, void* cuda_stream) {
  if (!h) return 1;
  if (!masks || !mixed_spec || !separated) return fail(h, "avsep_separate: null buffer");
  if (B < 1 || T < 1) return fail(h, "avsep_separate: B and T must be >= 1");
  CUDA_OK(cudaSetDevice(h->cfg.device));
  const char* e = launch_separate(static_cast<cudaStream_t>(cuda_stream), masks, mixed_spec, separated, B,
                                  h->cfg.num_speakers, h->cfg.freq_bins, T, lengths);
  return e ? fail(h, e) : 0;
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
  if (!h) return 1;
  FlagSet f;
  if (make_flag_set(h, flags, n, f, "avsep_flag_signal")) return 1;
  CUDA_OK(cudaSetDevice(h->cfg.device));
  const char* e = launch_flag_signal(static_cast<cudaStream_t>(cuda_stream), f, value);
  return e ? fail(h, e) : 0;
}

int avsep_flag_wait(avsep_handle* h, uint32_t* const* flags, int32_t n, uint32_t value, double timeout_s,
                    void* cuda_stream) {
  if (!h) return 1;
  FlagSet f;
  if (make_flag_set(h, flags, n, f, "avsep_flag_wait")) return 1;
  if (!(timeout_s > 0.0) || timeout_s > 3600.0) return fail(h, "avsep_flag_wait: timeout_s must be in (0, 3600]");
  CUDA_OK(cudaSetDevice(h->cfg.device));
  const char* e = launch_flag_wait(static_cast<cudaStream_t>(cuda_stream), f, value, timeout_s);
  return e ? fail(h, e) : 0;
}

// ---- sub-module forwards ------------------------------------------------------------------------
int avsep_audio_encoder(avsep_handle* h, const float* mixed_spec, int32_t B, int32_t T, float* out_BTd,
                        void* cuda_stream) {
  if (!h) return 1;
  if (!mixed_spec || !out_BTd) return fail(h, "avsep_audio_encoder: null buffer");
  if (check_shape(h, B, T, 1, 1, 1)) return 1;
  CUDA_OK(cudaSetDevice(h->cfg.device));
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  Workspace w;
  if (get_workspace(h, w, nullptr, 0, B, T, 1, 1, 1)) return 1;
  const int d = h->cfg.d_model, Ma = B * T;
  h->launches = 0;
  if (audio_frontend(h, s, w, mixed_spec, Plan{})) return 1;
  if (encoder_stack(h, s, h->enc_a, B, T, w.x_a, w.y_a, w.a_op, w.qkv_a, w.attn_a, w.ffn_a, nullptr, nullptr)) return 1;
  CUDA_OK(cudaMemcpyAsync(out_BTd, w.x_a, static_cast<size_t>(Ma) * d * 4, cudaMemcpyDeviceToDevice, s));
  return 0;
}

int avsep_visual_encoder(avsep_handle* h, const float* lip_frames, int32_t B, int32_t N, int32_t Hh, int32_t Ww,
                         int32_t target_len, float* out_BTd, void* cuda_stream) {
  if (!h) return 1;
  if (!lip_frames || !out_BTd) return fail(h, "avsep_visual_encoder: null buffer");
  if (check_shape(h, B, 1, N, Hh, Ww)) return 1;
  if (target_len < 1) return fail(h, "avsep_visual_encoder: target_len must be >= 1");
  CUDA_OK(cudaSetDevice(h->cfg.device));
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  Workspace w;
  if (get_workspace(h, w, nullptr, 0, B, 1, N, Hh, Ww)) return 1;
  const int d = h->cfg.d_model;
  h->launches = 0;
  if (visual_frontend(h, s, w, lip_frames, Plan{})) return 1;
  if (encoder_stack(h, s, h->enc_v, B, N, w.x_v, w.y_v, w.v_op, w.qkv_v, w.attn_v, w.ffn_v, nullptr, nullptr)) return 1;
  interp_rows_kernel<<<dim3(target_len, B), 128, 0, s>>>(w.x_v, out_BTd, N, target_len, d,
                                                         static_cast<float>(N) / static_cast<float>(target_len));
  CUDA_OK(cudaGetLastError());
  ++h->launches;
  return 0;
}

int avsep_fusion(avsep_handle* h, const float* audio_BTd, const float* visual_BLd, int32_t B, int32_t T, int32_t L,
                 float* out_BTd, void* cuda_stream) {
  if (!h) return 1;
  if (!audio_BTd || !visual_BLd || !out_BTd) return fail(h, "avsep_fusion: null buffer");
  if (check_shape(h, B, T, L, 1, 1)) return 1;
  if (L != T) return fail(h, "avsep_fusion: audio and visual must have the same length (model.py:131-133)");
  CUDA_OK(cudaSetDevice(h->cfg.device));
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  Workspace w;
  if (get_workspace(h, w, nullptr, 0, B, T, L, 1, 1)) return 1;
  const int d = h->cfg.d_model, Ma = B * T, Mv = B * L, prec = h->cfg.precision;
  h->launches = 0;
  CUDA_OK(cudaMemcpyAsync(w.x_a, audio_BTd, static_cast<size_t>(Ma) * d * 4, cudaMemcpyDeviceToDevice, s));
  CKL("add_layernorm", launch_add_layernorm(s, prec, w.x_a, nullptr, h->fus[0].n1g, h->fus[0].n1b, nullptr, w.a_op, Ma, d));
  CKL("add_layernorm", launch_add_layernorm(s, prec, visual_BLd, nullptr, nullptr, nullptr, nullptr, w.v_op, Mv, d));   // cast only
  const bool dbg = h->debug;
  h->debug = false;
  const int rc = fusion_stack(h, s, w, L);   // identity interpolation (L == T)
  h->debug = dbg;
  if (rc) return 1;
  // fused rows in fp32: recompute the final LayerNorm from the fp32 residual stream straight into the caller's buffer
  CKL("add_layernorm", launch_add_layernorm(s, PREC_TF32, w.x_a, nullptr, h->fng, h->fnb, nullptr, out_BTd, Ma, d));
  return 0;
}

int avsep_decoder(avsep_handle* h, const float* fused_BTd, const float* mixed_spec, int32_t B, int32_t T,
                  float* separated, float* masks, void* cuda_stream) {
  if (!h) return 1;
  if (!fused_BTd || !mixed_spec || !separated || !masks) return fail(h, "avsep_decoder: null buffer");
  if (check_shape(h, B, T, 1, 1, 1)) return 1;
  CUDA_OK(cudaSetDevice(h->cfg.device));
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  Workspace w;
  if (get_workspace(h, w, nullptr, 0, B, T, 1, 1, 1)) return 1;
  const int d = h->cfg.d_model, Ma = B * T;
  h->launches = 0;
  CKL("add_layernorm", launch_add_layernorm(s, h->cfg.precision, fused_BTd, nullptr, nullptr, nullptr, nullptr, w.a_op, Ma, d));
  return decoder_stage(h, s, w, mixed_spec, separated, masks);
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
  *count = it->second.second;
  if (host_out == nullptr) return 0;
  if (capacity < it->second.second) return fail(h, "avsep_debug_get_stage: buffer too small");
  CUDA_OK(cudaDeviceSynchronize());
  CUDA_OK(cudaMemcpy(host_out, it->second.first, it->second.second * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

int avsep_set_profile(avsep_handle* h, int32_t enable) {
  if (!h) return 1;
  h->profile = enable != 0;
  pdl_set(h->pdl && !h->profile);   // per-launch event pairs measure kernels one at a time
  return 0;
}

// Folds the pending event pairs into the per-label totals (synchronises) and writes
// "label count total_ms\n" lines into buf.  reset != 0 clears the totals afterwards.
int avsep_profile_report(avsep_handle* h, char* buf, size_t capacity, int32_t reset) {
  if (!h || !buf || capacity == 0) return fail(h, "avsep_profile_report: bad argument");
  CUDA_OK(cudaDeviceSynchronize());
  for (auto& mk : h->ev_marks) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev_pool[mk.second], h->ev_pool[mk.second + 1]) == cudaSuccess) {
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
  if (!h) return 1;
  const GemmProblem p = dense(A, M, K, W, N);
  GemmEpilogue e;
  e.bias = bias; e.act = act; e.out_f32 = out; e.ld_f32 = N;
  CK(launch_gemm(static_cast<cudaStream_t>(cuda_stream), h->cfg.precision, p, e, h->num_sms, force_bn));
  return 0;
}

// out-proj/FFN2-style GEMM with the fused residual + LayerNorm epilogue: x (in/out, fp32 [M,N]) += A W^T + bias;
// out_op = LN_{gamma,beta}(x) in operand precision.
int avsep_test_gemm_ln(avsep_handle* h, const void* A, const void* W, const float* bias, float* x, const float* gamma,
                       const float* beta, void* out_op, int32_t M, int32_t N, int32_t K, void* cuda_stream) {
  if (!h) return 1;
  const GemmProblem p = dense(A, M, K, W, N);
  GemmEpilogue e;
  e.kind = EPI_LN;
  e.bias = bias; e.resid = x; e.out_f32 = x; e.ld_f32 = N; e.ln_gamma = gamma; e.ln_beta = beta;
  e.out_op = out_op; e.ld_op = N;
  CK(launch_gemm(static_cast<cudaStream_t>(cuda_stream), h->cfg.precision, p, e, h->num_sms));
  return 0;
}

// Debug: same GEMM as avsep_test_gemm / avsep_test_gemm_ln (ln != 0) with a per-CTA phase trace:
// trace_dev[cta*8 + k] = globaltimer (ns) at k = 0 entry, 1 setup done, 2 first operands landed, 3 MMAs issued,
// 4 accumulator ready, 5 accumulator drained (LN), 6 first tile's epilogue done, 7 CTA done.
int avsep_test_gemm_trace(avsep_handle* h, const void* A, const void* W, const float* bias, float* x_or_out,
                          const float* gamma, const float* beta, void* out_op, int32_t M, int32_t N, int32_t K,
                          int32_t ln, int32_t act, unsigned long long* trace_dev, void* cuda_stream) {
  if (!h) return 1;
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
  CK(launch_gemm(static_cast<cudaStream_t>(cuda_stream), h->cfg.precision, p, e, h->num_sms, 0, trace_dev));
  return 0;
}

// Fused FFN sub-layer (d_model = 256, bf16): x (fp32, in place) += W2 act(W1 a + b1) + b2; out_op = LN(x) (bf16).
int avsep_test_ffn_fused(avsep_handle* h, const void* a, const void* w1, const float* b1, const void* w2,
                         const float* b2, int32_t act, float* x_inout, const float* gamma, const float* beta,
                         void* out_op, int32_t M, void* cuda_stream) {
  if (!h) return 1;
  CK(launch_ffn_fused(static_cast<cudaStream_t>(cuda_stream), a, w1, b1, w2, b2, act,
                                                             x_inout, x_inout, gamma, beta, out_op, M, h->num_sms, nullptr));
  return 0;
}

// Debug: the same with a phase trace ([grid][64] globaltimer stamps of each CTA's first tile: [0] entry, [1] A landed,
// [2] acc2 complete, [3] epilogue-2 done, per chunk j at 8+4j: GEMM1 issued, GEMM2 issued, acc1 ready, H published).
int avsep_test_ffn_fused_trace(avsep_handle* h, const void* a, const void* w1, const float* b1, const void* w2,
                               const float* b2, int32_t act, float* x_inout, const float* gamma, const float* beta,
                               void* out_op, int32_t M, unsigned long long* trace_dev, void* cuda_stream) {
  if (!h) return 1;
  CK(launch_ffn_fused(static_cast<cudaStream_t>(cuda_stream), a, w1, b1, w2, b2, act,
                                                             x_inout, x_inout, gamma, beta, out_op, M, h->num_sms, trace_dev));
  return 0;
}

// One whole stack through the fused kernel (xformer_stack_sm100.cu) on the handle's weights.  which: 0 audio encoder,
// 1 visual encoder, 2 fusion (kv = bf16 [B*L, num_fusion_layers*2*d] K|V rows).  x_in fp32 [B*L, d]; out_x fp32 and /
// or out_op bf16 (final_ln != 0: the LayerNorm that follows the stack in the model -- fusion layer 0 norm1 after the
// audio encoder, fusion.norm after the fusion stack; the visual encoder has none -- else a plain cast).
int avsep_test_xformer_stack(avsep_handle* h, int32_t which, const float* x_in, const void* kv, int32_t B, int32_t L,
                             float* out_x, void* out_op, int32_t final_ln, long long* trace_dev, void* cuda_stream) {
  if (!h) return 1;
  if (!h->finalized) return fail(h, "weights not finalized");
  if (which < 0 || which > 2) return fail(h, "test_xformer_stack: which must be 0, 1 or 2");
  if (h->xs_a == nullptr || !xformer_stack_usable(h->cfg.precision, h->cfg.d_model, h->cfg.nhead, L))
    return fail(h, "test_xformer_stack: the fused stack kernel does not support this configuration");
  StackProblem sp{};
  sp.x_in = x_in; sp.out_x = out_x; sp.out_op = out_op; sp.kv = kv; sp.B = B; sp.L = L; sp.trace = trace_dev;
  if (final_ln && which == 0) { sp.fin_gamma = h->fus[0].n1g; sp.fin_beta = h->fus[0].n1b; }
  if (final_ln && which == 2) { sp.fin_gamma = h->fng; sp.fin_beta = h->fnb; }
  h->prof_stream = static_cast<cudaStream_t>(cuda_stream);
  return run_stack(h, static_cast<cudaStream_t>(cuda_stream), which, sp);
}

int avsep_test_fusion_decoder(avsep_handle* h, const float* x_in, const void* kv, int32_t B, int32_t L, const float* mixed,
                              float* separated, float* masks, long long* trace_dev, void* cuda_stream) {
  if (!h) return 1;
  if (!h->finalized) return fail(h, "weights not finalized");
  if (h->xs_f == nullptr || !h->xs_f_decoder || !xformer_stack_usable(h->cfg.precision, h->cfg.d_model, h->cfg.nhead, L))
    return fail(h, "test_fusion_decoder: the fused stack kernel does not support this configuration");
  if (!mixed || !separated || !masks) return fail(h, "test_fusion_decoder: null buffer");
  StackProblem sp{};
  sp.x_in = x_in; sp.fin_gamma = h->fng; sp.fin_beta = h->fnb; sp.kv = kv; sp.B = B; sp.L = L; sp.trace = trace_dev;
  sp.mixed = mixed; sp.separated = separated; sp.masks = masks;
  h->prof_stream = static_cast<cudaStream_t>(cuda_stream);
  return run_stack(h, static_cast<cudaStream_t>(cuda_stream), 2, sp);
}

int avsep_set_option(avsep_handle* h, const char* name, int32_t value) {
  if (!h || !name) return 1;
  if (strcmp(name, "host_chunk") == 0) { h->host_chunk = value; return 0; }
  if (strcmp(name, "host_lanes") == 0) { h->host_lanes = value; return 0; }
  if (strcmp(name, "pdl") == 0) { h->pdl = value != 0; pdl_set(h->pdl && !h->profile); drop_graphs(h); return 0; }
  if (strcmp(name, "use_graph") == 0) { h->use_graph = value != 0; return 0; }
  if (strcmp(name, "two_stream") == 0) { h->two_stream = value != 0; drop_graphs(h); return 0; }
  if (strcmp(name, "attn_tc") == 0) { h->attn_tc = value; drop_graphs(h); return 0; }
  if (strcmp(name, "profile_spin_us") == 0) { h->profile_spin_us = value; return 0; }
  return fail(h, std::string("unknown option ") + name);
}

int avsep_test_conv1d(avsep_handle* h, const void* A_padded, const void* W3, const float* bias, float* out, int32_t B,
                      int32_t L, int32_t N, int32_t K, void* cuda_stream) {
  if (!h) return 1;
  GemmProblem p{};
  const int Mp = B * (L + 2);
  p.A = A_padded; p.lda = K; p.rowsA = Mp; p.M = Mp; p.W = W3; p.ldw = 3 * K; p.N = N; p.K = K;
  p.taps = 3; p.tap_stride = K; p.row_shift = -1;
  GemmEpilogue e;
  e.bias = bias; e.rowmap = ROW_PAD2COMPACT; e.Lp = L + 2; e.out_f32 = out; e.ld_f32 = N;
  CK(launch_gemm(static_cast<cudaStream_t>(cuda_stream), h->cfg.precision, p, e, h->num_sms));
  return 0;
}

int avsep_test_attention(avsep_handle* h, const void* q, const void* k, const void* v, void* out, int32_t B, int32_t H,
                         int32_t hd, int32_t Lq, int32_t Lk, int32_t lerp_src, void* cuda_stream) {
  if (!h) return 1;
  AttnProblem ap{};
  ap.q = q; ap.ldq = H * hd; ap.k = k; ap.v = v; ap.ldkv = H * hd; ap.out = out; ap.ldo = H * hd;
  ap.B = B; ap.H = H; ap.hd = hd; ap.Lq = Lq; ap.Lk = Lk; ap.lerp_src = lerp_src; ap.tc_mode = h->attn_tc;
  cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
  void* scratch = nullptr;
  if (lerp_src > 0) {   // same routing as fusion_stack: K then V columns side by side in one interpolated buffer
    AttnProblem tp = ap;
    tp.lerp_src = 0; tp.ldkv = 2 * H * hd;
    if (attention_tc_wanted(h->cfg.precision, tp)) {
      const int dm = H * hd;
      if (cudaMalloc(&scratch, static_cast<size_t>(B) * Lk * 2 * dm * 2) != cudaSuccess) return fail(h, "test_attention: cudaMalloc failed");
      tp.k = scratch; tp.v = static_cast<__nv_bfloat16*>(scratch) + dm;
      CK(launch_lerp_rows(s, static_cast<const float*>(k), dm, B, lerp_src, Lk, dm, scratch, 2 * dm));
      CK(launch_lerp_rows(s, static_cast<const float*>(v), dm, B, lerp_src, Lk, dm, static_cast<__nv_bfloat16*>(scratch) + dm, 2 * dm));
      ap = tp;
    }
  }
  const char* err = launch_attention(s, h->cfg.precision, ap);
  if (scratch) { cudaStreamSynchronize(s); cudaFree(scratch); }
  if (err) return fail(h, err);
  return 0;
}

int avsep_test_add_layernorm(avsep_handle* h, const float* x, const float* y, const float* gamma, const float* beta,
                             float* x_out, void* out_op, int32_t M, int32_t d, void* cuda_stream) {
  if (!h) return 1;
  CKL("add_layernorm", launch_add_layernorm(static_cast<cudaStream_t>(cuda_stream), h->cfg.precision, x, y, gamma, beta, x_out, out_op, M, d));
  return 0;
}

int avsep_test_visual_cnn(avsep_handle* h, const float* frames, int32_t M, int32_t Hh, int32_t Ww, void* pooled,
                          void* cuda_stream) {
  if (!h) return 1;
  if (!h->finalized) return fail(h, "weights not finalized");
  CK(run_visual_cnn(h, static_cast<cudaStream_t>(cuda_stream), frames, M, Hh, Ww, pooled));
  return 0;
}

// Debug: tcgen05 CNN with a phase trace ([grid][64] globaltimer stamps of each CTA's second frame group).
int avsep_test_visual_cnn_trace(avsep_handle* h, const float* frames, int32_t M, void* pooled,
                                unsigned long long* trace_dev, void* cuda_stream) {
  if (!h) return 1;
  if (!h->finalized) return fail(h, "weights not finalized");
  CK(run_visual_cnn(h, static_cast<cudaStream_t>(cuda_stream), frames, M, 32, 32, pooled, trace_dev));
  return 0;
}

}  // extern "C"
