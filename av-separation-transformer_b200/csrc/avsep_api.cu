// C-ABI layer of libavsep.so (see include/avsep.h): handle, weight prepack, workspace plan and the forward
// orchestration of AVSeparationTransformer.forward (reference: model.py:268-276 and everything it calls).
#include "../../include/avsep.h"
#include "kernels.h"

#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

using namespace avsep;

namespace {

std::string g_create_error;

inline uint16_t f2bf_host(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return static_cast<uint16_t>(u >> 16);
}

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

struct EncLayerW {
  const void *wqkv, *wo, *w1, *w2;
  const float *bqkv, *bo, *b1, *b2, *n1g, *n1b, *n2g, *n2b;
};
struct FusLayerW {
  const void *wq, *wo, *w1, *w2;
  const float *bq, *bo, *b1, *b2, *n1g, *n1b, *n2g, *n2b;
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
  std::vector<EncLayerW> enc_a, enc_v;
  std::vector<FusLayerW> fus;
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

int linear(avsep_handle* h, cudaStream_t s, const char* label, const void* A, int M, int K, const void* W,
           const float* bias, int N, int act, float* out_f32, void* out_op) {
  GemmProblem p{};
  p.A = A; p.lda = K; p.rowsA = M; p.M = M; p.W = W; p.ldw = K; p.N = N; p.K = K;
  p.taps = 1; p.tap_stride = 0; p.row_shift = 0;
  GemmEpilogue e;
  e.bias = bias; e.act = act;
  // a GELU whose only consumer is a bf16 operand does not need the fp32-grade erf
  if (act == ACT_GELU && h->cfg.precision == AVSEP_PREC_BF16 && out_f32 == nullptr) e.act = ACT_GELU_BF16;
  e.out_f32 = out_f32; e.ld_f32 = N;
  e.out_op = out_op; e.ld_op = N;
  CKL(label, launch_gemm(s, h->cfg.precision, p, e));
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
    CKL(label, launch_gemm(s, prec, p, e));
    return 0;
  }
  e.kind = EPI_STD;
  e.out_op = nullptr;
  if (resid != nullptr) {
    e.out_f32 = y; e.ld_f32 = p.N;
    CKL(label, launch_gemm(s, prec, p, e));
    CKL("add_layernorm", launch_add_layernorm(s, prec, resid, y, g, b, x_out, out_op, rows_out, p.N));
  } else {
    e.out_f32 = x_out; e.ld_f32 = p.N;
    CKL(label, launch_gemm(s, prec, p, e));
    CKL("add_layernorm", launch_add_layernorm(s, prec, x_out, nullptr, g, b, nullptr, out_op, rows_out, p.N));
  }
  return 0;
}

int linear_resid_ln(avsep_handle* h, cudaStream_t s, const char* label, const void* A, int M, int K, const void* W,
                    const float* bias, int N, float* x, const float* g, const float* b, void* out_op, float* y) {
  GemmProblem p{};
  p.A = A; p.lda = K; p.rowsA = M; p.M = M; p.W = W; p.ldw = K; p.N = N; p.K = K; p.taps = 1;
  GemmEpilogue e;
  e.bias = bias;
  return gemm_resid_ln(h, s, label, p, e, x, x, g, b, out_op, M, y);
}

bool stack_fusable(const avsep_handle* h, int len) {
  return h->xs_a != nullptr && xformer_stack_usable(h->cfg.precision, h->cfg.d_model, h->cfg.nhead, len);
}

// A whole stack in one kernel (xformer_stack_sm100.cu).  which: 0 audio encoder, 1 visual encoder, 2 fusion.
int run_stack(avsep_handle* h, cudaStream_t s, int which, const float* x_in, float* out_x, void* out_op,
              const float* fin_g, const float* fin_b, const void* kv, int kv_ld, int B, int L, long long* trace = nullptr,
              const float* mixed = nullptr, float* separated = nullptr, float* masks = nullptr, const void* pro_a = nullptr,
              void* kvp_out = nullptr, int kvp_L = 0, const int* lens = nullptr, const int* kvp_lens = nullptr) {
  StackProblem sp{};
  sp.trace = trace;
  sp.lens = lens; sp.kvp_lens = kvp_lens;
  if (kvp_out != nullptr) {      // which 1: the fusion layers' K | V rows are produced inside the kernel
    sp.kvp_out = kvp_out; sp.kvp_L = kvp_L; sp.kvp_n = h->cfg.num_fusion_layers * 2 * h->cfg.d_model; sp.kvp_ld = sp.kvp_n;
  }
  if (pro_a != nullptr) {        // x_in is produced inside the kernel (which 0: Conv1d #2 + ReLU + PE; 1: frame_proj + PE)
    sp.pro_a = pro_a; sp.pro_relu = which == 0;
    sp.pro_taps = which == 0 ? 3 : 1; sp.pro_k = which == 0 ? h->cfg.d_model : 128;
    sp.pro_pitch = which == 0 ? L + 2 : L; sp.pro_rows = B * sp.pro_pitch;
    sp.pe = which == 0 ? h->pe_a : h->pe_v;
  }
  sp.mixed = mixed; sp.separated = separated; sp.masks = masks; sp.F = h->cfg.freq_bins; sp.S = h->cfg.num_speakers;
  sp.x_in = x_in; sp.out_x = out_x; sp.out_op = out_op; sp.fin_gamma = fin_g; sp.fin_beta = fin_b;
  sp.wstream = which == 0 ? (pro_a ? h->xs_a : h->xs_a_np) : which == 1 ? (pro_a ? h->xs_v : h->xs_v_np) : h->xs_f;
  sp.n_layers = which == 2 ? h->cfg.num_fusion_layers : h->cfg.num_encoder_layers;
  sp.cross = which == 2;
  sp.kv = kv; sp.kv_ld = kv_ld;
  sp.B = B; sp.L = L;
  sp.act = which == 2 ? ACT_GELU : ACT_RELU;
  CKL(which == 0 ? "layer.audio_enc" : which == 1 ? "layer.visual_enc" : masks ? "layer.fusion_decoder" : "layer.fusion",
      launch_xformer_stack(s, sp, h->num_sms));
  return 0;
}

// One fused kernel per feed-forward sub-layer (ffn_fused_sm100.cu) from this many rows on; below it the unfused GEMM
// pair spreads over more CTAs and wins.
constexpr int FFN_FUSED_MIN_ROWS = 2048;

// nn.TransformerEncoderLayer x L (pre-norm, ReLU FFN; model.py:48-52,59; torch transformer.py:946-950).
// In: x (fp32 residual stream), a_op = LN_{layer0.norm1}(x).  Out: x, a_op = LN_{final}(x) (or cast when final_g == null).
// lens: keys per utterance of a variable-length batch, or null.
int encoder_stack(avsep_handle* h, cudaStream_t s, const std::vector<EncLayerW>& layers, int B, int L, float* x,
                  float* y, void* a_op, void* qkv, void* attn, void* ffn, const float* final_g, const float* final_b,
                  const int* lens = nullptr) {
  const int d = h->cfg.d_model, H = h->cfg.nhead, M = B * L, prec = h->cfg.precision;
  const size_t os = op_size(h);
  for (size_t l = 0; l < layers.size(); ++l) {
    const EncLayerW& w = layers[l];
    if (linear(h, s, "gemm.qkv", a_op, M, d, w.wqkv, w.bqkv, 3 * d, ACT_NONE, nullptr, qkv)) return 1;
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
    const float* g = last ? final_g : layers[l + 1].n1g;
    const float* b = last ? final_b : layers[l + 1].n1b;
    if (ffn_fusable(prec, d) && M >= FFN_FUSED_MIN_ROWS) {
      CKL("ffn.fused", launch_ffn_fused(s, a_op, w.w1, w.b1, w.w2, w.b2, ACT_RELU, x, x,
                                                                             g, b, a_op, M, h->num_sms, nullptr));
    } else {
      if (linear(h, s, "gemm.ffn1", a_op, M, d, w.w1, w.b1, 4 * d, ACT_RELU, nullptr, ffn)) return 1;
      if (linear_resid_ln(h, s, "gemm.ffn2", ffn, M, 4 * d, w.w2, w.b2, d, x, g, b, a_op, y)) return 1;
    }
  }
  return 0;
}

// AudioEncoder up to (not including) the transformer: Conv1d+ReLU x2, +PE (model.py:56-58), then the first
// layer's LayerNorm: x_a (fp32) and a_op = LN_{g,b}(x_a).
// x_only: the fused stack kernel computes the first LayerNorm itself, so only the fp32 residual rows are written.
int audio_frontend(avsep_handle* h, cudaStream_t s, Workspace& w, const float* mixed, const float* g, const float* b,
                   bool x_only = false, bool conv1_only = false) {
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
    CKL("gemm.conv1d_0", launch_gemm(s, prec, p, e));
  }
  if (conv1_only) return 0;      // Conv1d #2 + ReLU + PE run inside the encoder stack kernel, on h1
  {
    GemmProblem p{};
    p.A = w.h1; p.lda = d; p.rowsA = Map; p.M = Map; p.W = h->wc2; p.ldw = 3 * d; p.N = d; p.K = d;
    p.taps = 3; p.tap_stride = d; p.row_shift = -1;
    GemmEpilogue e;
    e.bias = h->bc2; e.act = ACT_RELU; e.rowmap = ROW_PAD2COMPACT; e.Lp = T + 2;
    e.pe = h->pe_a;
    if (x_only) {
      e.out_f32 = w.x_a; e.ld_f32 = d;
      CKL("gemm.conv1d_2", launch_gemm(s, prec, p, e));
    } else if (gemm_resid_ln(h, s, "gemm.conv1d_2", p, e, nullptr, w.x_a, g, b, w.a_op, B * T, w.y_a)) {
      return 1;
    }
  }
  return snapshot(h, s, "audio_embed", w.x_a, static_cast<size_t>(B) * T * d, false);
}

// VisualEncoder up to (not including) the transformer: CNN, pool, frame_proj, +PE (model.py:106-110), then the
// first layer's LayerNorm: x_v (fp32) and v_op = LN_{g,b}(x_v).
int visual_frontend(avsep_handle* h, cudaStream_t s, Workspace& w, const float* frames, const float* g, const float* b,
                    bool x_only = false, bool cnn_only = false) {
  h->prof_stream = s;
  const int d = h->cfg.d_model, B = w.B, N = w.N;
  const int Mv = B * N;
  CKL("visual_cnn", run_visual_cnn(h, s, frames, Mv, w.Hh, w.Ww, w.pooled, nullptr, w.frame_lens, N));
  if (snapshot(h, s, "visual_pool", w.pooled, static_cast<size_t>(Mv) * 128, true)) return 1;
  if (cnn_only) return 0;        // frame_proj + PE run inside the encoder stack kernel, on the pooled features
  GemmProblem p{};
  p.A = w.pooled; p.lda = 128; p.rowsA = Mv; p.M = Mv; p.W = h->wproj; p.ldw = 128; p.N = d; p.K = 128;
  p.taps = 1;
  GemmEpilogue e;
  e.bias = h->bproj; e.pe = h->pe_v; e.pe_period = N;
  if (x_only) {
    e.out_f32 = w.x_v; e.ld_f32 = d;
    CKL("gemm.frame_proj", launch_gemm(s, h->cfg.precision, p, e));
  } else if (gemm_resid_ln(h, s, "gemm.frame_proj", p, e, nullptr, w.x_v, g, b, w.v_op, Mv, w.y_v)) {
    return 1;
  }
  return snapshot(h, s, "visual_embed", w.x_v, static_cast<size_t>(Mv) * d, false);
}

// CrossModalFusion (model.py:145-149,166-173).  In: x_a residual stream, a_op = LN_{layer0.norm1}(x_a),
// v_op = visual rows (L_src per utterance).  Out: a_op = fusion.norm(x) in operand precision.
// Fused variant (stack_fusable(T)): the visual rows are interpolated to the audio frame rate first, exactly where the
// reference does it (model.py:114-116, before the K/V projection), the K|V rows of every fusion layer come from one GEMM
// on those T rows (bf16), and the whole fusion stack runs in one kernel.  In: x_a (fp32 residual), x_v (fp32 visual
// encoder output, L_src rows per utterance).  Out: a_op = fusion.norm(x) in bf16.
// with_decoder (out: *decoded = true): SeparationDecoder runs inside the same kernel and writes separated / masks.
int fusion_stack_fused(avsep_handle* h, cudaStream_t s, Workspace& w, int L_src, const float* mixed, float* separated,
                       float* masks, bool* decoded, bool have_kv = false) {
  h->prof_stream = s;
  const int d = h->cfg.d_model, B = w.B, T = w.T;
  const int Ma = B * T, Lf = h->cfg.num_fusion_layers;
  if (!have_kv) {                // else the visual stack kernel has already written w.kvb
    CKL("lerp_kv", launch_lerp_rows(s, w.x_v, d, B, L_src, T, d, w.attn_a, d, w.frame_lens, w.lens));
    if (linear(h, s, "gemm.cross_kv", w.attn_a, Ma, d, h->wkv_all, h->bkv_all, Lf * 2 * d, ACT_NONE, nullptr, w.kvb)) return 1;
  }
  *decoded = h->xs_f_decoder && !h->debug && masks != nullptr;
  if (*decoded)
    return run_stack(h, s, 2, w.x_a, nullptr, nullptr, h->fng, h->fnb, w.kvb, Lf * 2 * d, B, T, nullptr, mixed, separated, masks,
                     nullptr, nullptr, 0, w.lens);
  if (run_stack(h, s, 2, w.x_a, h->debug ? w.x_a : nullptr, w.a_op, h->fng, h->fnb, w.kvb, Lf * 2 * d, B, T, nullptr, nullptr,
                nullptr, nullptr, nullptr, nullptr, 0, w.lens))
    return 1;
  return snapshot(h, s, "fused", w.a_op, static_cast<size_t>(Ma) * d, true);
}

int fusion_stack(avsep_handle* h, cudaStream_t s, Workspace& w, int L_src) {
  h->prof_stream = s;
  const int d = h->cfg.d_model, H = h->cfg.nhead, B = w.B, T = w.T, prec = h->cfg.precision;
  const int Ma = B * T, Mv = B * L_src, Lf = h->cfg.num_fusion_layers;
  // K/V projection of every fusion layer in one GEMM on the un-interpolated visual rows
  if (linear(h, s, "gemm.cross_kv", w.v_op, Mv, d, h->wkv_all, h->bkv_all, Lf * 2 * d, ACT_NONE, w.kvn, nullptr)) return 1;
  for (int l = 0; l < Lf; ++l) {
    const FusLayerW& fw = h->fus[l];
    if (linear(h, s, "gemm.cross_q", w.a_op, Ma, d, fw.wq, fw.bq, d, ACT_NONE, nullptr, w.qkv_a)) return 1;
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
    const float* g = last ? h->fng : h->fus[l + 1].n1g;
    const float* b = last ? h->fnb : h->fus[l + 1].n1b;
    if (ffn_fusable(prec, d) && Ma >= FFN_FUSED_MIN_ROWS) {
      CKL("ffn.fused", launch_ffn_fused(s, w.a_op, fw.w1, fw.b1, fw.w2, fw.b2, ACT_GELU,
                                                                             w.x_a, w.x_a, g, b, w.a_op, Ma, h->num_sms,
                                                                             nullptr));
    } else {
      if (linear(h, s, "gemm.ffn1", w.a_op, Ma, d, fw.w1, fw.b1, 4 * d, ACT_GELU, nullptr, w.ffn_a)) return 1;
      if (linear_resid_ln(h, s, "gemm.ffn2", w.ffn_a, Ma, 4 * d, fw.w2, fw.b2, d, w.x_a, g, b, w.a_op, w.y_a)) return 1;
    }
  }
  return snapshot(h, s, "fused", w.a_op, static_cast<size_t>(Ma) * d, true);
}

// SeparationDecoder.forward + .separate (model.py:201-220): a_op = fused rows in operand precision.
int decoder_stage(avsep_handle* h, cudaStream_t s, Workspace& w, const float* mixed, float* separated, float* masks) {
  h->prof_stream = s;
  const int d = h->cfg.d_model, F = h->cfg.freq_bins, S = h->cfg.num_speakers, B = w.B, T = w.T;
  const int Ma = B * T;
  if (linear(h, s, "gemm.dec0", w.a_op, Ma, d, h->wdec0, h->bdec0, 2 * d, ACT_GELU, nullptr, w.ffn_a)) return 1;
  GemmProblem p{};
  p.A = w.ffn_a; p.lda = 2 * d; p.rowsA = Ma; p.M = Ma; p.W = h->wdec3; p.ldw = 2 * d; p.N = S * F; p.K = 2 * d;
  p.taps = 1;
  GemmEpilogue e;
  e.kind = EPI_TAIL;
  e.bias = h->bdec3;
  e.mixed = mixed; e.masks = masks; e.separated = separated; e.F = F; e.S = S; e.T = T;
  e.lens = w.lens;
  CKL("gemm.dec3_tail", launch_gemm(s, h->cfg.precision, p, e));
  return 0;
}

int forward_device(avsep_handle* h, cudaStream_t s, Workspace& w, const float* mixed, const float* frames,
                   float* separated, float* masks) {
  const int d = h->cfg.d_model;
  const int Ma = w.B * w.T, Mv = w.B * w.N;
  h->prof_stream = s;
  if (h->profile && h->profile_spin_us > 0) spin_kernel<<<1, 1, 0, s>>>(1000ull * h->profile_spin_us);
  // The audio and visual branches are independent until the fusion: run them on two streams (fork / join) unless
  // per-kernel profiling or stage snapshots need a single ordered stream.
  cudaStream_t sv = s;
  const bool fork = h->two_stream && !h->profile && !h->debug;
  if (fork) {
    if (h->aux_stream == nullptr) {
      CUDA_OK(cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
      CUDA_OK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
      CUDA_OK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    }
    sv = h->aux_stream;
    CUDA_OK(cudaEventRecord(h->ev_fork, s));
    CUDA_OK(cudaStreamWaitEvent(sv, h->ev_fork, 0));
  }
  const bool fa = stack_fusable(h, w.T), fv = stack_fusable(h, w.N);
  const bool ff = fa && fv;            // the fused fusion stack reads the fp32 residual rows of both encoders
  // --- visual branch (enqueued first: its CNN is the longest kernel) ---
  const bool fp = !h->debug;     // input projections inside the stack kernels (no stage snapshots then)
  bool kvp = false;
  if (visual_frontend(h, sv, w, frames, h->enc_v[0].n1g, h->enc_v[0].n1b, fv, fv && fp)) return 1;
  if (fv) {
    // out: x_v (fp32) for the interpolation in front of the K/V projection; v_op (bf16 cast) only for the unfused fusion
    // fused K | V projection: needs the fused fusion stack behind it and the audio frames inside a visual tile slot
    kvp = ff && h->xs_v_kvp && !h->debug &&
          xformer_kvp_usable(h->cfg.num_fusion_layers * 2 * d, w.N, w.T);
    if (run_stack(h, sv, 1, w.x_v, kvp ? nullptr : w.x_v, (ff || kvp) ? nullptr : w.v_op, nullptr, nullptr, nullptr, 0, w.B,
                  w.N, nullptr, nullptr, nullptr, nullptr, fp ? w.pooled : nullptr, kvp ? w.kvb : nullptr, w.T, w.frame_lens,
                  w.lens))
      return 1;
  } else if (encoder_stack(h, sv, h->enc_v, w.B, w.N, w.x_v, w.y_v, w.v_op, w.qkv_v, w.attn_v, w.ffn_v, nullptr, nullptr,
                           w.frame_lens)) {
    return 1;
  }
  if (snapshot(h, sv, "visual_enc", w.x_v, static_cast<size_t>(Mv) * d, false)) return 1;
  // --- audio branch ---
  if (audio_frontend(h, s, w, mixed, h->enc_a[0].n1g, h->enc_a[0].n1b, fa, fa && fp)) return 1;
  if (fa) {
    if (run_stack(h, s, 0, w.x_a, w.x_a, ff ? nullptr : w.a_op, h->fus[0].n1g, h->fus[0].n1b, nullptr, 0, w.B, w.T, nullptr,
                  nullptr, nullptr, nullptr, fp ? w.h1 : nullptr, nullptr, 0, w.lens))
      return 1;
  } else if (encoder_stack(h, s, h->enc_a, w.B, w.T, w.x_a, w.y_a, w.a_op, w.qkv_a, w.attn_a, w.ffn_a, h->fus[0].n1g,
                           h->fus[0].n1b, w.lens)) {
    return 1;
  }
  if (snapshot(h, s, "audio_enc", w.x_a, static_cast<size_t>(Ma) * d, false)) return 1;
  if (fork) {
    CUDA_OK(cudaEventRecord(h->ev_join, sv));
    CUDA_OK(cudaStreamWaitEvent(s, h->ev_join, 0));
  }
  // --- fusion + decoder ---
  if (ff) {
    bool decoded = false;
    if (fusion_stack_fused(h, s, w, w.N, mixed, separated, masks, &decoded, kvp)) return 1;
    if (decoded) return 0;
  } else if (fusion_stack(h, s, w, w.N)) {
    return 1;
  }
  return decoder_stage(h, s, w, mixed, separated, masks);
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

struct ArenaBuilder {
  std::vector<uint8_t> bytes;
  size_t add(const void* src, size_t n) {
    const size_t off = align_up(bytes.size(), 256);
    bytes.resize(off + n);
    if (src) memcpy(bytes.data() + off, src, n);
    return off;
  }
  size_t add_f32(const float* src, size_t n) { return add(src, n * 4); }
  size_t add_op(const float* src, size_t n, bool tf32) {
    if (tf32) {   // round to tf32 (10-bit mantissa, nearest, ties away) so the tensor core's truncation is exact
      std::vector<float> tmp(n);
      for (size_t i = 0; i < n; ++i) {
        uint32_t u;
        memcpy(&u, &src[i], 4);
        if ((u & 0x7f800000u) != 0x7f800000u) u = (u + 0x1000u) & 0xffffe000u;
        memcpy(&tmp[i], &u, 4);
      }
      return add(tmp.data(), n * 4);
    }
    std::vector<uint16_t> tmp(n);
    for (size_t i = 0; i < n; ++i) tmp[i] = f2bf_host(src[i]);
    return add(tmp.data(), n * 2);
  }
};

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
  if (const char* e = gemm_init()) return fail(nullptr, e);
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
  ArenaBuilder ar;
  std::map<std::string, size_t> off;
#define GETW(var, key, ...)                                  \
  const HostTensor* var = find_w(h, key, {__VA_ARGS__});     \
  if (!var) return 1;

  // --- AudioEncoder Conv1d weights: (Cout, Cin, 3) -> (Cout, 3*Cin_pad), k = tap*Cin_pad + c
  {
    GETW(w0, "audio_encoder.input_proj.0.weight", d, F, 3);
    GETW(b0, "audio_encoder.input_proj.0.bias", d);
    GETW(w2, "audio_encoder.input_proj.2.weight", d, d, 3);
    GETW(b2, "audio_encoder.input_proj.2.bias", d);
    std::vector<float> p0(static_cast<size_t>(d) * 3 * Fp, 0.f), p2(static_cast<size_t>(d) * 3 * d, 0.f);
    for (int64_t o = 0; o < d; ++o)
      for (int64_t c = 0; c < F; ++c)
        for (int tap = 0; tap < 3; ++tap) p0[(o * 3 + tap) * Fp + c] = w0->data[(o * F + c) * 3 + tap];
    for (int64_t o = 0; o < d; ++o)
      for (int64_t c = 0; c < d; ++c)
        for (int tap = 0; tap < 3; ++tap) p2[(o * 3 + tap) * d + c] = w2->data[(o * d + c) * 3 + tap];
    off["wc1"] = ar.add_op(p0.data(), p0.size(), tf32);
    off["wc2"] = ar.add_op(p2.data(), p2.size(), tf32);
    off["bc1"] = ar.add_f32(b0->data.data(), d);
    off["bc2"] = ar.add_f32(b2->data.data(), d);
    GETW(pea, "audio_encoder.pos_enc.pe", 1, 5000, d);
    GETW(pev, "visual_encoder.pos_enc.pe", 1, 5000, d);
    off["pe_a"] = ar.add_f32(pea->data.data(), pea->data.size());
    off["pe_v"] = ar.add_f32(pev->data.data(), pev->data.size());
  }
  // --- encoder stacks
  for (int stack = 0; stack < 2; ++stack) {
    const std::string pre = stack == 0 ? "audio_encoder" : "visual_encoder";
    for (int l = 0; l < Le; ++l) {
      const std::string p = pre + ".transformer.layers." + std::to_string(l);
      const std::string t = (stack == 0 ? "a" : "v") + std::to_string(l);
      GETW(wqkv, p + ".self_attn.in_proj_weight", 3 * d, d);
      GETW(bqkv, p + ".self_attn.in_proj_bias", 3 * d);
      GETW(wo, p + ".self_attn.out_proj.weight", d, d);
      GETW(bo, p + ".self_attn.out_proj.bias", d);
      GETW(w1, p + ".linear1.weight", 4 * d, d);
      GETW(b1, p + ".linear1.bias", 4 * d);
      GETW(w2, p + ".linear2.weight", d, 4 * d);
      GETW(b2, p + ".linear2.bias", d);
      GETW(n1g, p + ".norm1.weight", d);
      GETW(n1b, p + ".norm1.bias", d);
      GETW(n2g, p + ".norm2.weight", d);
      GETW(n2b, p + ".norm2.bias", d);
      off[t + "wqkv"] = ar.add_op(wqkv->data.data(), wqkv->data.size(), tf32);
      off[t + "wo"] = ar.add_op(wo->data.data(), wo->data.size(), tf32);
      off[t + "w1"] = ar.add_op(w1->data.data(), w1->data.size(), tf32);
      off[t + "w2"] = ar.add_op(w2->data.data(), w2->data.size(), tf32);
      off[t + "bqkv"] = ar.add_f32(bqkv->data.data(), 3 * d);
      off[t + "bo"] = ar.add_f32(bo->data.data(), d);
      off[t + "b1"] = ar.add_f32(b1->data.data(), 4 * d);
      off[t + "b2"] = ar.add_f32(b2->data.data(), d);
      off[t + "n1g"] = ar.add_f32(n1g->data.data(), d);
      off[t + "n1b"] = ar.add_f32(n1b->data.data(), d);
      off[t + "n2g"] = ar.add_f32(n2g->data.data(), d);
      off[t + "n2b"] = ar.add_f32(n2b->data.data(), d);
    }
  }
  // --- VisualEncoder CNN: fold BatchNorm (eval) into conv weight/bias, repack tap-major, fragment order
  {
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
    std::vector<uint32_t> p1(visual_cnn_pack_sizes(1)), p2(visual_cnn_pack_sizes(2)), p3(visual_cnn_pack_sizes(3));
    visual_cnn_pack(folded[0].data(), folded[1].data(), folded[2].data(), p1.data(), p2.data(), p3.data());
    std::vector<uint8_t> tc2(visual_cnn_tc_w2_bytes()), tc3(visual_cnn_tc_w3_bytes());
    visual_cnn_tc_pack(folded[1].data(), folded[2].data(), tc2.data(), tc3.data());
    off["tcw2"] = ar.add(tc2.data(), tc2.size());
    off["tcw3"] = ar.add(tc3.data(), tc3.size());
    off["cw1"] = ar.add(p1.data(), p1.size() * 4);
    off["cw2"] = ar.add(p2.data(), p2.size() * 4);
    off["cw3"] = ar.add(p3.data(), p3.size() * 4);
    visual_cnn_pack(folded[0].data(), folded[1].data(), folded[2].data(), p1.data(), p2.data(), p3.data(), true);
    off["cw1l"] = ar.add(p1.data(), p1.size() * 4);
    off["cw2l"] = ar.add(p2.data(), p2.size() * 4);
    off["cw3l"] = ar.add(p3.data(), p3.size() * 4);
    off["cb1"] = ar.add_f32(fbias[0].data(), 32);
    off["cb2"] = ar.add_f32(fbias[1].data(), 64);
    off["cb3"] = ar.add_f32(fbias[2].data(), 128);
    GETW(wp, "visual_encoder.frame_proj.weight", d, 128);
    GETW(bp_, "visual_encoder.frame_proj.bias", d);
    off["wproj"] = ar.add_op(wp->data.data(), wp->data.size(), tf32);
    off["bproj"] = ar.add_f32(bp_->data.data(), d);
  }
  // --- fusion: q rows of the packed in_proj per layer; k|v rows of every layer concatenated
  {
    std::vector<float> wkv(static_cast<size_t>(Lf) * 2 * d * d), bkv(static_cast<size_t>(Lf) * 2 * d);
    for (int l = 0; l < Lf; ++l) {
      const std::string p = "fusion.layers." + std::to_string(l);
      const std::string t = "f" + std::to_string(l);
      GETW(win, p + ".cross_attn.in_proj_weight", 3 * d, d);
      GETW(bin, p + ".cross_attn.in_proj_bias", 3 * d);
      GETW(wo, p + ".cross_attn.out_proj.weight", d, d);
      GETW(bo, p + ".cross_attn.out_proj.bias", d);
      GETW(w1, p + ".ff.0.weight", 4 * d, d);
      GETW(b1, p + ".ff.0.bias", 4 * d);
      GETW(w2, p + ".ff.3.weight", d, 4 * d);
      GETW(b2, p + ".ff.3.bias", d);
      GETW(n1g, p + ".norm1.weight", d);
      GETW(n1b, p + ".norm1.bias", d);
      GETW(n2g, p + ".norm2.weight", d);
      GETW(n2b, p + ".norm2.bias", d);
      off[t + "wq"] = ar.add_op(win->data.data(), static_cast<size_t>(d) * d, tf32);
      off[t + "bq"] = ar.add_f32(bin->data.data(), d);
      memcpy(wkv.data() + static_cast<size_t>(l) * 2 * d * d, win->data.data() + d * d, sizeof(float) * 2 * d * d);
      memcpy(bkv.data() + static_cast<size_t>(l) * 2 * d, bin->data.data() + d, sizeof(float) * 2 * d);
      off[t + "wo"] = ar.add_op(wo->data.data(), wo->data.size(), tf32);
      off[t + "w1"] = ar.add_op(w1->data.data(), w1->data.size(), tf32);
      off[t + "w2"] = ar.add_op(w2->data.data(), w2->data.size(), tf32);
      off[t + "bo"] = ar.add_f32(bo->data.data(), d);
      off[t + "b1"] = ar.add_f32(b1->data.data(), 4 * d);
      off[t + "b2"] = ar.add_f32(b2->data.data(), d);
      off[t + "n1g"] = ar.add_f32(n1g->data.data(), d);
      off[t + "n1b"] = ar.add_f32(n1b->data.data(), d);
      off[t + "n2g"] = ar.add_f32(n2g->data.data(), d);
      off[t + "n2b"] = ar.add_f32(n2b->data.data(), d);
    }
    off["wkv"] = ar.add_op(wkv.data(), wkv.size(), tf32);
    off["bkv"] = ar.add_f32(bkv.data(), bkv.size());
    GETW(fg, "fusion.norm.weight", d);
    GETW(fb, "fusion.norm.bias", d);
    off["fng"] = ar.add_f32(fg->data.data(), d);
    off["fnb"] = ar.add_f32(fb->data.data(), d);
  }
  // --- decoder
  {
    GETW(w0, "decoder.decoder.0.weight", 2 * d, d);
    GETW(b0, "decoder.decoder.0.bias", 2 * d);
    GETW(w3, "decoder.decoder.3.weight", S * F, 2 * d);
    GETW(b3, "decoder.decoder.3.bias", S * F);
    off["wdec0"] = ar.add_op(w0->data.data(), w0->data.size(), tf32);
    off["wdec3"] = ar.add_op(w3->data.data(), w3->data.size(), tf32);
    off["bdec0"] = ar.add_f32(b0->data.data(), 2 * d);
    off["bdec3"] = ar.add_f32(b3->data.data(), S * F);
  }
  // --- fused transformer-stack kernel: weight streams in consumption order + per-layer vector blocks
  const bool pack_stacks = xformer_stack_usable(h->cfg.precision, static_cast<int>(d), h->cfg.nhead, 1);
  if (pack_stacks) {
    const size_t vf = static_cast<size_t>(xformer_vec_floats());
    for (int stack = 0; stack < 2; ++stack) {
      const std::string pre = stack == 0 ? "audio_encoder" : "visual_encoder";
      // the stream starts with the input projection (Conv1d #2 as 3 taps x 256 / frame_proj as 1 x 128), whose bias
      // rides in layer 0's vector block
      const size_t pro_bytes = stack == 0 ? xformer_pro_bytes(3, static_cast<int>(d)) : xformer_pro_bytes(1, 128);
      const int n_kv = static_cast<int>(Lf * 2 * d);
      const bool with_kvp = stack == 1 && xformer_kvp_usable(n_kv, 1, 1);
      std::vector<uint8_t> stream(pro_bytes + static_cast<size_t>(Le) * xformer_stream_bytes(false) +
                                  (with_kvp ? xformer_kvp_bytes(n_kv) : 0));
      const HostTensor* b0t = nullptr;
      if (stack == 0) {
        GETW(wc, "audio_encoder.input_proj.2.weight", d, d, 3);
        GETW(bc, "audio_encoder.input_proj.2.bias", d);
        xformer_pack_pro(wc->data.data(), static_cast<int>(3 * d), 3, 3, static_cast<int>(d), stream.data());
        b0t = bc;
      } else {
        GETW(wc, "visual_encoder.frame_proj.weight", d, 128);
        GETW(bc, "visual_encoder.frame_proj.bias", d);
        xformer_pack_pro(wc->data.data(), 128, 1, 1, 128, stream.data());
        b0t = bc;
      }
      std::vector<float> vecs(vf);
      for (int l = 0; l < Le; ++l) {
        const std::string p = pre + ".transformer.layers." + std::to_string(l);
        GETW(wqkv, p + ".self_attn.in_proj_weight", 3 * d, d);
        GETW(bqkv, p + ".self_attn.in_proj_bias", 3 * d);
        GETW(wo, p + ".self_attn.out_proj.weight", d, d);
        GETW(bo, p + ".self_attn.out_proj.bias", d);
        GETW(w1, p + ".linear1.weight", 4 * d, d);
        GETW(b1, p + ".linear1.bias", 4 * d);
        GETW(w2, p + ".linear2.weight", d, 4 * d);
        GETW(b2, p + ".linear2.bias", d);
        GETW(n1g, p + ".norm1.weight", d);
        GETW(n1b, p + ".norm1.bias", d);
        GETW(n2g, p + ".norm2.weight", d);
        GETW(n2b, p + ".norm2.bias", d);
        xformer_pack_vecs(bqkv->data.data(), static_cast<int>(3 * d), bo->data.data(), b1->data.data(), b2->data.data(),
                          n1g->data.data(), n1b->data.data(), n2g->data.data(), n2b->data.data(), vecs.data(),
                          l == 0 ? b0t->data.data() : nullptr);
        xformer_pack_self(wqkv->data.data(), wo->data.data(), w1->data.data(), w2->data.data(), vecs.data(),
                          stream.data() + pro_bytes + static_cast<size_t>(l) * xformer_stream_bytes(false));
      }
      if (with_kvp) {
        std::vector<float> wkv(static_cast<size_t>(n_kv) * d), bkv(n_kv);
        for (int l = 0; l < Lf; ++l) {
          const std::string p = "fusion.layers." + std::to_string(l);
          GETW(win, p + ".cross_attn.in_proj_weight", 3 * d, d);
          GETW(bin, p + ".cross_attn.in_proj_bias", 3 * d);
          memcpy(wkv.data() + static_cast<size_t>(l) * 2 * d * d, win->data.data() + d * d, sizeof(float) * 2 * d * d);
          memcpy(bkv.data() + static_cast<size_t>(l) * 2 * d, bin->data.data() + d, sizeof(float) * 2 * d);
        }
        xformer_pack_kvp(wkv.data(), bkv.data(), n_kv, stream.data() + pro_bytes + static_cast<size_t>(Le) * xformer_stream_bytes(false));
        h->xs_v_kvp = true;
      }
      off[stack == 0 ? "xs_a" : "xs_v"] = ar.add(stream.data(), stream.size());
    }
    const bool fuse_dec = xformer_decoder_usable(static_cast<int>(S), static_cast<int>(F));
    std::vector<uint8_t> stream(static_cast<size_t>(Lf) * xformer_stream_bytes(true) +
                                (fuse_dec ? xformer_decoder_bytes(static_cast<int>(S), static_cast<int>(F)) : 0));
    std::vector<float> vecs(vf);
    for (int l = 0; l < Lf; ++l) {
      const std::string p = "fusion.layers." + std::to_string(l);
      GETW(win, p + ".cross_attn.in_proj_weight", 3 * d, d);
      GETW(bin, p + ".cross_attn.in_proj_bias", 3 * d);
      GETW(wo, p + ".cross_attn.out_proj.weight", d, d);
      GETW(bo, p + ".cross_attn.out_proj.bias", d);
      GETW(w1, p + ".ff.0.weight", 4 * d, d);
      GETW(b1, p + ".ff.0.bias", 4 * d);
      GETW(w2, p + ".ff.3.weight", d, 4 * d);
      GETW(b2, p + ".ff.3.bias", d);
      GETW(n1g, p + ".norm1.weight", d);
      GETW(n1b, p + ".norm1.bias", d);
      GETW(n2g, p + ".norm2.weight", d);
      GETW(n2b, p + ".norm2.bias", d);
      xformer_pack_vecs(bin->data.data(), static_cast<int>(d), bo->data.data(), b1->data.data(), b2->data.data(),
                        n1g->data.data(), n1b->data.data(), n2g->data.data(), n2b->data.data(), vecs.data());
      xformer_pack_cross(win->data.data(), wo->data.data(), w1->data.data(), w2->data.data(), vecs.data(),
                         stream.data() + static_cast<size_t>(l) * xformer_stream_bytes(true));
    }
    if (fuse_dec) {
      GETW(w0, "decoder.decoder.0.weight", 2 * d, d);
      GETW(b0, "decoder.decoder.0.bias", 2 * d);
      GETW(w3, "decoder.decoder.3.weight", S * F, 2 * d);
      GETW(b3, "decoder.decoder.3.bias", S * F);
      xformer_pack_decoder(w0->data.data(), b0->data.data(), w3->data.data(), b3->data.data(), static_cast<int>(S), static_cast<int>(F),
                           stream.data() + static_cast<size_t>(Lf) * xformer_stream_bytes(true));
    }
    h->xs_f_decoder = fuse_dec;
    off["xs_f"] = ar.add(stream.data(), stream.size());
  }
#undef GETW
  // upload
  drop_graphs(h);
  if (h->d_weights) cudaFree(h->d_weights);
  h->d_weights = nullptr;
  CUDA_OK(cudaMalloc(&h->d_weights, ar.bytes.size()));
  h->weight_bytes = ar.bytes.size();
  CUDA_OK(cudaMemcpyAsync(h->d_weights, ar.bytes.data(), ar.bytes.size(), cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaStreamSynchronize(s));
  auto P = [&](const std::string& k) -> const void* { return h->d_weights + off.at(k); };
  auto PF = [&](const std::string& k) -> const float* { return reinterpret_cast<const float*>(h->d_weights + off.at(k)); };
  h->wc1 = P("wc1"); h->wc2 = P("wc2"); h->bc1 = PF("bc1"); h->bc2 = PF("bc2");
  h->pe_a = PF("pe_a"); h->pe_v = PF("pe_v");
  h->wproj = P("wproj"); h->bproj = PF("bproj");
  h->wkv_all = P("wkv"); h->bkv_all = PF("bkv"); h->fng = PF("fng"); h->fnb = PF("fnb");
  h->wdec0 = P("wdec0"); h->wdec3 = P("wdec3"); h->bdec0 = PF("bdec0"); h->bdec3 = PF("bdec3");
  h->cnn.w1 = reinterpret_cast<const uint32_t*>(P("cw1")); h->cnn.b1 = PF("cb1");
  h->cnn.w2 = reinterpret_cast<const uint32_t*>(P("cw2")); h->cnn.b2 = PF("cb2");
  h->cnn.w3 = reinterpret_cast<const uint32_t*>(P("cw3")); h->cnn.b3 = PF("cb3");
  h->cnn.w1l = reinterpret_cast<const uint32_t*>(P("cw1l"));
  h->cnn.w2l = reinterpret_cast<const uint32_t*>(P("cw2l"));
  h->cnn.w3l = reinterpret_cast<const uint32_t*>(P("cw3l"));
  h->cnn_w2_slabs = static_cast<const uint8_t*>(P("tcw2"));
  h->cnn_w3_rows = static_cast<const uint8_t*>(P("tcw3"));
  h->xs_a = h->xs_v = h->xs_f = nullptr;
  if (pack_stacks) {
    h->xs_a = static_cast<const uint8_t*>(P("xs_a")); h->xs_v = static_cast<const uint8_t*>(P("xs_v"));
    h->xs_a_np = h->xs_a + xformer_pro_bytes(3, h->cfg.d_model); h->xs_v_np = h->xs_v + xformer_pro_bytes(1, 128);
    h->xs_f = static_cast<const uint8_t*>(P("xs_f"));
  }
  h->enc_a.clear(); h->enc_v.clear(); h->fus.clear();
  for (int stack = 0; stack < 2; ++stack)
    for (int l = 0; l < Le; ++l) {
      const std::string t = (stack == 0 ? "a" : "v") + std::to_string(l);
      EncLayerW w;
      w.wqkv = P(t + "wqkv"); w.wo = P(t + "wo"); w.w1 = P(t + "w1"); w.w2 = P(t + "w2");
      w.bqkv = PF(t + "bqkv"); w.bo = PF(t + "bo"); w.b1 = PF(t + "b1"); w.b2 = PF(t + "b2");
      w.n1g = PF(t + "n1g"); w.n1b = PF(t + "n1b"); w.n2g = PF(t + "n2g"); w.n2b = PF(t + "n2b");
      (stack == 0 ? h->enc_a : h->enc_v).push_back(w);
    }
  for (int l = 0; l < Lf; ++l) {
    const std::string t = "f" + std::to_string(l);
    FusLayerW w;
    w.wq = P(t + "wq"); w.wo = P(t + "wo"); w.w1 = P(t + "w1"); w.w2 = P(t + "w2");
    w.bq = PF(t + "bq"); w.bo = PF(t + "bo"); w.b1 = PF(t + "b1"); w.b2 = PF(t + "b2");
    w.n1g = PF(t + "n1g"); w.n1b = PF(t + "n1b"); w.n2g = PF(t + "n2g"); w.n2b = PF(t + "n2b");
    h->fus.push_back(w);
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
  if (!h) return 1;
  if (!waves || !spec) return fail(h, "avsep_stft: null argument");
  CUDA_OK(cudaSetDevice(h->cfg.device));
  CK(launch_stft_complex(static_cast<cudaStream_t>(cuda_stream), waves, B, L, n_fft, hop_length, spec, mag));
  h->launches = 1;
  return 0;
}

int avsep_istft(avsep_handle* h, const float* spec, const float* masks, int32_t B, int32_t S, int32_t T,
                int32_t n_fft, int32_t hop_length, int32_t L, float* waves, void* cuda_stream) {
  if (!h) return 1;
  if (!spec || !waves) return fail(h, "avsep_istft: null argument");
  CUDA_OK(cudaSetDevice(h->cfg.device));
  CK(launch_istft_masked(static_cast<cudaStream_t>(cuda_stream), spec, masks, B, S, T, n_fft, hop_length, L, waves));
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
  if (!h) return 1;
  if (!masks || !mixed_spec || !separated) return fail(h, "avsep_separate: null buffer");
  if (B < 1 || T < 1) return fail(h, "avsep_separate: B and T must be >= 1");
  CUDA_OK(cudaSetDevice(h->cfg.device));
  const char* e = launch_separate(static_cast<cudaStream_t>(cuda_stream), masks, mixed_spec, separated, B,
                                  h->cfg.num_speakers, h->cfg.freq_bins, T);
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
  if (audio_frontend(h, s, w, mixed_spec, h->enc_a[0].n1g, h->enc_a[0].n1b)) return 1;
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
  if (visual_frontend(h, s, w, lip_frames, h->enc_v[0].n1g, h->enc_v[0].n1b)) return 1;
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
  const int save_prec = h->cfg.precision;
  CKL("add_layernorm", launch_add_layernorm(s, PREC_TF32, w.x_a, nullptr, h->fng, h->fnb, nullptr, out_BTd, Ma, d));
  (void)save_prec;
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
  GemmProblem p{};
  p.A = A; p.lda = K; p.rowsA = M; p.M = M; p.W = W; p.ldw = K; p.N = N; p.K = K; p.taps = 1;
  GemmEpilogue e;
  e.bias = bias; e.act = act; e.out_f32 = out; e.ld_f32 = N;
  CK(launch_gemm(static_cast<cudaStream_t>(cuda_stream), h->cfg.precision, p, e, force_bn));
  return 0;
}

// out-proj/FFN2-style GEMM with the fused residual + LayerNorm epilogue: x (in/out, fp32 [M,N]) += A W^T + bias;
// out_op = LN_{gamma,beta}(x) in operand precision.
int avsep_test_gemm_ln(avsep_handle* h, const void* A, const void* W, const float* bias, float* x, const float* gamma,
                       const float* beta, void* out_op, int32_t M, int32_t N, int32_t K, void* cuda_stream) {
  if (!h) return 1;
  GemmProblem p{};
  p.A = A; p.lda = K; p.rowsA = M; p.M = M; p.W = W; p.ldw = K; p.N = N; p.K = K; p.taps = 1;
  GemmEpilogue e;
  e.kind = EPI_LN;
  e.bias = bias; e.resid = x; e.out_f32 = x; e.ld_f32 = N; e.ln_gamma = gamma; e.ln_beta = beta;
  e.out_op = out_op; e.ld_op = N;
  CK(launch_gemm(static_cast<cudaStream_t>(cuda_stream), h->cfg.precision, p, e));
  return 0;
}

// Debug: same GEMM as avsep_test_gemm / avsep_test_gemm_ln (ln != 0) with a per-CTA phase trace:
// trace_dev[cta*8 + k] = globaltimer (ns) at k = 0 entry, 1 setup done, 2 first operands landed, 3 MMAs issued,
// 4 accumulator ready, 5 accumulator drained (LN), 6 first tile's epilogue done, 7 CTA done.
int avsep_test_gemm_trace(avsep_handle* h, const void* A, const void* W, const float* bias, float* x_or_out,
                          const float* gamma, const float* beta, void* out_op, int32_t M, int32_t N, int32_t K,
                          int32_t ln, int32_t act, unsigned long long* trace_dev, void* cuda_stream) {
  if (!h) return 1;
  GemmProblem p{};
  p.A = A; p.lda = K; p.rowsA = M; p.M = M; p.W = W; p.ldw = K; p.N = N; p.K = K; p.taps = 1;
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
  CK(launch_gemm(static_cast<cudaStream_t>(cuda_stream), h->cfg.precision, p, e, 0, trace_dev));
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
  const float *g = nullptr, *b = nullptr;
  if (final_ln && which == 0) { g = h->fus[0].n1g; b = h->fus[0].n1b; }
  if (final_ln && which == 2) { g = h->fng; b = h->fnb; }
  h->prof_stream = static_cast<cudaStream_t>(cuda_stream);
  return run_stack(h, static_cast<cudaStream_t>(cuda_stream), which, x_in, out_x, out_op, g, b, kv,
                   h->cfg.num_fusion_layers * 2 * h->cfg.d_model, B, L, trace_dev);
}

int avsep_test_fusion_decoder(avsep_handle* h, const float* x_in, const void* kv, int32_t B, int32_t L, const float* mixed,
                              float* separated, float* masks, long long* trace_dev, void* cuda_stream) {
  if (!h) return 1;
  if (!h->finalized) return fail(h, "weights not finalized");
  if (h->xs_f == nullptr || !h->xs_f_decoder || !xformer_stack_usable(h->cfg.precision, h->cfg.d_model, h->cfg.nhead, L))
    return fail(h, "test_fusion_decoder: the fused stack kernel does not support this configuration");
  if (!mixed || !separated || !masks) return fail(h, "test_fusion_decoder: null buffer");
  h->prof_stream = static_cast<cudaStream_t>(cuda_stream);
  return run_stack(h, static_cast<cudaStream_t>(cuda_stream), 2, x_in, nullptr, nullptr, h->fng, h->fnb, kv,
                   h->cfg.num_fusion_layers * 2 * h->cfg.d_model, B, L, trace_dev, mixed, separated, masks);
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
  CK(launch_gemm(static_cast<cudaStream_t>(cuda_stream), h->cfg.precision, p, e));
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
