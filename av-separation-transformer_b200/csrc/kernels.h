// Internal (C++) interface between the C-ABI layer (avsep_api.cu) and the sm_100a kernels.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <string.h>

namespace avsep {

// fp32 -> bf16 bit pattern, round to nearest even as __float2bfloat16_rn (NaN stays a quiet NaN): every host-side
// weight packer rounds through this one function, so all uploaded bf16 weights agree with the device conversion.
inline uint16_t f2bf(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return static_cast<uint16_t>(u >> 16);
}

// ---- host helpers of the launchers (launch_util.cu); the const char* functions return nullptr or a static error ----
// Resolves cuTensorMapEncodeTiled from the driver; called once by avsep_create before any launcher runs.
const char* tma_init();
// TMA descriptor of a row-major [outer, inner] tensor with leading dimension ld_elems (elements of esz bytes), moved in
// boxes of box_outer rows x box_inner elements: 128-byte swizzle, 256-byte L2 promotion, out-of-range elements read as
// zero and not written.  The pointer must be 16-byte aligned and the row pitch a multiple of 16 bytes.
const char* tma_encode_2d(CUtensorMap* map, CUtensorMapDataType dt, int esz, const void* ptr, uint64_t inner,
                          uint64_t outer, uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer);
// The same for `batches` such tensors stored back to back ([batches, outer, inner]); a box stays inside one batch.
const char* tma_encode_3d(CUtensorMap* map, CUtensorMapDataType dt, int esz, const void* ptr, uint64_t inner,
                          uint64_t outer, uint64_t batches, uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer);
// Raises the kernel's dynamic shared-memory limit on the current device to `bytes` unless this process already set it
// at least that high there (up to 48 KB needs no opt-in).  False when the runtime refuses.
bool smem_opt_in(const void* kern, int bytes);
template <typename... KArgs>
bool smem_opt_in(void (*kern)(KArgs...), int bytes) {
  return smem_opt_in(reinterpret_cast<const void*>(kern), bytes);
}

// Where a forward-path kernel runs: its stream, and whether it may use programmatic dependent launch (PDL).  Every
// kernel launched through launch_pdl calls griddep_wait() before it touches anything its predecessor wrote, so
// pdl = false only means plain stream order.  The launching handle decides (its "pdl" option, off while it profiles).
struct LaunchCtx {
  cudaStream_t stream;
  bool pdl;
};
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, LaunchCtx lc, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = lc.stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = lc.pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}


enum Precision { PREC_BF16 = 0, PREC_TF32 = 1 };
enum Act { ACT_NONE = 0, ACT_RELU = 1, ACT_GELU = 2, ACT_GELU_BF16 = 3 };   // 3: erf-GELU to bf16 accuracy (polynomial)
// How accumulator row m of the GEMM maps to an output row.
//   ROW_IDENT       out row = m
//   ROW_PAD2PAD     rows live in a per-utterance padded space of Lp = L+2 rows (zero halo row on each side,
//                   the Conv1d zero padding); out row = m, halo rows are written as zeros
//   ROW_PAD2COMPACT padded space in, compact (B*L) rows out; halo rows are dropped
enum RowMap { ROW_IDENT = 0, ROW_PAD2PAD = 1, ROW_PAD2COMPACT = 2 };
// EPI_LN_TMA and EPI_TAIL_MASKS (EPI_TAIL with separated == null) are selected internally by launch_gemm
enum EpiKind { EPI_STD = 0, EPI_TAIL = 1, EPI_LN = 2, EPI_LN_TMA = 3, EPI_TAIL_MASKS = 4 };

struct GemmProblem {
  const void* A;   // [rowsA, K] K-major activations (bf16 or fp32/tf32), leading dimension lda (elements)
  int lda;
  int rowsA;       // rows that exist in A (TMA zero-fills outside)
  int M;           // accumulator rows to produce
  const void* W;   // [N, taps*tap_stride] K-major weights, leading dimension ldw
  int ldw;
  int N;
  int K;           // reduction length per tap
  int taps;        // 1 = plain GEMM, 3 = Conv1d(k=3) as three row-shifted passes into the same accumulator
  int tap_stride;  // column offset between taps in W
  int row_shift;   // A row offset of tap 0 relative to the accumulator row (-1 for padding=1)
};

struct GemmEpilogue {
  int kind = EPI_STD;
  const float* bias = nullptr;   // [N]
  int act = ACT_NONE;
  int rowmap = ROW_IDENT;
  int Lp = 0;                    // padded rows per utterance for the PAD modes
  const float* pe = nullptr;     // positional table [max_len, N] added after the activation
  int pe_period = 0;             // ROW_IDENT: position = m % pe_period
  float* out_f32 = nullptr;      // fp32 output (residual-stream precision), leading dimension ld_f32
  int ld_f32 = 0;
  void* out_op = nullptr;        // operand-precision output (bf16, or fp32 in the tf32 path) for the next GEMM
  int ld_op = 0;
  // EPI_LN: value (bias/act/PE/rowmap as above) + resid -> out_f32 (fp32 residual stream, may alias resid), then
  // LayerNorm(ln_gamma, ln_beta, eps 1e-5) of the full row -> out_op.  ln_gamma == nullptr: out_op = plain cast.
  const float* resid = nullptr;  // [rows, N] fp32, indexed by the OUTPUT row
  const float* ln_gamma = nullptr;
  const float* ln_beta = nullptr;
  // EPI_TAIL (SeparationDecoder head): masks = sigmoid(acc + bias) -> masks[b,s,f,t]; separated = masks * mixed[b,f,t].
  // separated == null: masks only, and mixed is never read (may be null).
  const float* mixed = nullptr;
  float* masks = nullptr;
  float* separated = nullptr;
  int F = 0, S = 0, T = 0;
  // Variable-length batch (null: every utterance has all its rows).  ROW_PAD2PAD: rows t >= lens[b] (t = padded row - 1)
  // are written as zeros like the halo rows.  EPI_TAIL: masks / separated are 0 for t >= lens[b] and mixed is not read
  // there.  Values are clamped to [1, rows per utterance].
  const int* lens = nullptr;
};
// Per-utterance length of a variable-length batch: lens[b] clamped to [1, L], or L when lens is null.
__device__ __forceinline__ int utt_len(const int* lens, int b, int L) {
  return lens == nullptr ? L : min(max(__ldg(lens + b), 1), L);
}
// Frame fr of N-frame utterances lies within the first lens[fr / N] frames of its utterance (always when lens is null).
__device__ __forceinline__ bool frame_live(const int* lens, int N, int fr) {
  return lens == nullptr || fr % N < utt_len(lens, fr / N, N);
}

// Linear interpolation of nsrc rows to ndst rows along time: F.interpolate(mode='linear', align_corners=False), i.e.
// ATen upsample_linear1d (model.py:114-116).  Every kernel that stretches rows takes its source rows and weights from
// lerp_tap, with the scale from lerp_scale resolved once per utterance, outside the per-element loops.
__host__ __device__ __forceinline__ float lerp_scale(int nsrc, int ndst) {
  return static_cast<float>(nsrc) / static_cast<float>(ndst);   // as ATen computes it
}
struct LerpTap {
  int i0, i1;       // target row = w0 * source row i0 + w1 * source row i1
  float w0, w1;
};
__device__ __forceinline__ LerpTap lerp_tap(int t, int nsrc, float scale) {
  const float sp = fmaxf(scale * (static_cast<float>(t) + 0.5f) - 0.5f, 0.0f);
  LerpTap k;
  k.i0 = static_cast<int>(sp);
  if (k.i0 > nsrc - 1) k.i0 = nsrc - 1;
  k.i1 = min(k.i0 + 1, nsrc - 1);
  k.w1 = sp - static_cast<float>(k.i0);
  k.w0 = 1.0f - k.w1;
  return k;
}

// Returns nullptr on success or a static error string.
const char* launch_gemm(LaunchCtx lc, int prec, const GemmProblem& p, const GemmEpilogue& e, int num_sms,
                        int force_bn = 0, unsigned long long* trace = nullptr);   // trace: [grid][8] globaltimer stamps (debug)
bool gemm_ln_fusable(int N);   // EPI_LN usable for this row width

// Fused FFN sub-layer (d_model = 256, bf16): x += W2 act(W1 a + b1) + b2 ; out_op = LayerNorm(x)  (ffn_fused_sm100.cu)
bool ffn_fusable(int prec, int d_model);
const char* launch_ffn_fused(LaunchCtx lc, const void* a, const void* w1, const float* b1, const void* w2,
                             const float* b2, int act, const float* resid, float* x_out, const float* gamma,
                             const float* beta, void* out_op, int M, int num_sms,
                             unsigned long long* trace = nullptr);
// A whole transformer stack in one persistent kernel (xformer_stack_sm100.cu): d_model = 256, 4 heads, bf16, sequences of
// at most 128 rows.  The residual tile stays in tensor memory through every layer; weights stream as prepacked images.
struct StackProblem {
  const float* x_in;        // [B*L, 256] fp32 residual stream
  float* out_x;             // [B*L, 256] fp32 residual after the stack (may alias x_in) or null
  void* out_op;             // [B*L, 256] bf16: final LayerNorm (fin_gamma/fin_beta) or plain cast (fin_gamma == null), or null
  const float *fin_gamma, *fin_beta;
  const uint8_t* wstream;   // n_layers x xformer_stream_bytes(cross): per layer a vector block, then the weight items
  int n_layers;
  bool cross;               // false: self-attention encoder layers (ReLU); true: cross-attention fusion layers (GELU)
  const void* kv;           // cross: bf16 [B*L, kv_ld] rows, layer l's K at columns [l*512, +256), V at [l*512+256, +256)
  int kv_ld;
  int B, L;
  int act;
  long long* trace = nullptr;   // optional [grid][256] clock64 stamps (debug)
  // SeparationDecoder fused behind the fusion stack (cross only; replaces out_x / out_op): the stream then continues with
  // xformer_decoder_bytes(S, F) of decoder items (xformer_pack_decoder)
  // Input projection fused in front of layer 0 (self stacks; replaces x_in): x = act(sum_tap A[utt * pro_pitch + t + tap]
  // W_tap^T + b0) + pe[t].  The stream then starts with xformer_pro_bytes(pro_taps, pro_k) of projection items.
  const void* pro_a = nullptr;           // bf16 [pro_rows, pro_k]
  int pro_rows = 0, pro_pitch = 0, pro_taps = 0, pro_k = 0, pro_relu = 0;
  const float* pe = nullptr;             // fp32 [>= L, 256]
  // K | V projection of the fusion layers fused behind the last layer (self stacks; replaces out_x / out_op): the
  // output rows, interpolated to kvp_L rows per utterance, times the kvp_n stacked K | V weight rows -> bf16
  // [B * kvp_L, kvp_ld]; the stream then ends with xformer_kvp_bytes(kvp_n) of items (xformer_pack_kvp)
  void* kvp_out = nullptr;
  int kvp_L = 0, kvp_n = 0, kvp_ld = 0;
  const float* mixed = nullptr;          // (B, F, L) fp32
  float *masks = nullptr, *separated = nullptr;   // (B, S, F, L) fp32
  int F = 0, S = 0;
  // Variable-length batch (null: all L).  lens[b]: rows of utterance b that are real; its keys past them are masked,
  // the fused decoder stores 0 there and the K | V interpolation reads lens[b] source rows.  kvp_lens[b]: the
  // interpolation target (null: all kvp_L).  L stays the slot pitch; values are clamped to [1, L] / [1, kvp_L].
  const int* lens = nullptr;
  const int* kvp_lens = nullptr;
};
bool xformer_decoder_usable(int S, int F);
int xformer_decoder_chunks(int S, int F);
size_t xformer_decoder_bytes(int S, int F);
void xformer_pack_decoder(const float* w0, const float* b0, const float* w3, const float* b3, int S, int F, uint8_t* dst);
size_t xformer_pro_bytes(int taps, int K);
// W element (n, tap, k) at W[n * ld + k * col_stride + tap]: Conv1d weight (out, in, 3): ld = 3 in, col_stride = 3
void xformer_pack_pro(const float* W, int ld, int col_stride, int taps, int K, uint8_t* dst);
bool xformer_kvp_usable(int n, int L_src, int L_out);
size_t xformer_kvp_bytes(int n);
void xformer_pack_kvp(const float* wkv, const float* bkv, int n, uint8_t* dst);   // wkv [n, 256] row-major, bkv [n]
bool xformer_stack_usable(int prec, int d_model, int nhead, int len);
size_t xformer_stream_bytes(bool cross);
int xformer_vec_floats();
void xformer_pack_self(const float* wqkv, const float* wo, const float* w1, const float* w2, const float* vecs,
                       uint8_t* dst);   // vecs: xformer_vec_floats() values from xformer_pack_vecs
void xformer_pack_cross(const float* wq, const float* wo, const float* w1, const float* w2, const float* vecs,
                        uint8_t* dst);
void xformer_pack_vecs(const float* bqkv, int n_bqkv, const float* bo, const float* b1, const float* b2, const float* n1g,
                       const float* n1b, const float* n2g, const float* n2b, float* dst, const float* b0 = nullptr);
const char* launch_xformer_stack(LaunchCtx lc, const StackProblem& p, int num_sms);

// x_out = x + y (y may be null); out = LayerNorm(x_out) * gamma + beta (skipped when gamma == null, then out = x_out).
// out_op is bf16 (PREC_BF16) or fp32 (PREC_TF32).
const char* launch_add_layernorm(LaunchCtx lc, int prec, const float* x, const float* y, const float* gamma,
                                 const float* beta, float* x_out, void* out_op, int M, int d);

// mixed (B,F,T) fp32 -> Xp (B, T+2, Fp) operand precision, zero halo rows and zero pad columns; lens (or null):
// rows t >= lens[b] are zero.
const char* launch_prep_audio(LaunchCtx lc, int prec, const float* mixed, void* xp, int B, int F, int T, int Fp,
                              const int* lens = nullptr);

// SeparationDecoder.separate (model.py:210-220): out[b,s,f,t] = masks[b,s,f,t] * mixed[b,f,t] (peer_gather.cu).
// lens (or null): out[b,s,f,t] = 0 for t >= lens[b] (clamped to [1, T]), where masks and mixed are not read.
const char* launch_separate(cudaStream_t s, const float* masks, const float* mixed, float* out, long long B, int S,
                            int F, int T, const int* lens = nullptr);
// Packed variable-length batches (packed_io.cu): utterances b0 .. b0 + B - 1 of a packed batch, whose blocks sit back to
// back behind those of utterances 0 .. b0 - 1 (offsets summed on the device from lens / flens, clamped as utt_len
// clamps; null = all T / all N).  unpack: mixed_p (F, T_b) and frames_p (N_b, hw) blocks -> the valid regions of the
// padded (B, F, T) / (B, N, hw) staging; pack: the valid regions of the padded (B, S, F, T) sep / masks -> their
// (S, F, T_b) blocks.  Nothing past the lengths is read or written.
const char* launch_unpack(LaunchCtx lc, const float* mixed_p, const float* frames_p, const int* lens,
                          const int* flens, int b0, int B, int F, int T, int N, int hw, float* mixed, float* frames);
const char* launch_pack(LaunchCtx lc, const float* sep, const float* masks, const int* lens, int b0, int B, int S,
                        int F, int T, float* sep_p, float* masks_p);
// Ticket flags of the masks-only gather: 32-bit words in this GPU's or a peer's memory, raised / awaited in stream order.
struct FlagSet {
  static constexpr int MAX = 16;
  unsigned* ptr[MAX];
  int n;
};
const char* launch_flag_signal(cudaStream_t s, const FlagSet& f, unsigned value);
const char* launch_flag_wait(cudaStream_t s, const FlagSet& f, unsigned value, double timeout_s);

struct AttnProblem {
  const void* q; int ldq;          // operand-precision rows [B*Lq, ldq], head h at columns h*hd
  const void* k; const void* v;    // self: operand precision rows [B*Lk, ldkv]; cross (lerp): fp32 rows [B*Nsrc, ldkv]
  int ldkv;
  void* out; int ldo;              // operand precision [B*Lq, ldo]
  int B, H, hd, Lq, Lk;
  int lerp_src;                    // 0 = plain; >0 = K/V hold lerp_src source rows per utterance, interpolated to Lk rows
  int tc_mode;                     // tcgen05 kernel: 0 = never, 1 = when min(Lq, Lk) >= 96, 2 = whenever usable
  // Variable-length batch (null: all Lk / all lerp_src).  k_lens[b]: keys of utterance b (the rest are masked; on the
  // lerp path also the interpolation target); src_lens[b]: its interpolation source rows.  Lk / lerp_src stay the row
  // pitch of the K/V buffers; values are clamped to [1, Lk] / [1, lerp_src].
  const int* k_lens = nullptr;
  const int* src_lens = nullptr;
};
const char* launch_attention(LaunchCtx lc, int prec, const AttnProblem& p);
// tcgen05 flash attention (attention_tc.cu): bf16, head dim 64, materialised K/V rows.  launch_attention dispatches
// to it by itself when attention_tc_wanted.
bool attention_tc_usable(int prec, const AttnProblem& p);
bool attention_tc_wanted(int prec, const AttnProblem& p);      // usable and selected by p.tc_mode
const char* launch_attention_tc(LaunchCtx lc, const AttnProblem& p);
// dst[b*L + t, 0:cols] (bf16) = linear interpolation (lerp_tap) of src rows [b*nsrc + i, 0:cols] (fp32), with the
// scale of each utterance's own lengths: src_lens[b] source rows interpolated to dst_lens[b] rows (null: nsrc / L).
// The rows past dst_lens[b] are finite filler.
const char* launch_lerp_rows(LaunchCtx lc, const float* src, int ld_src, int B, int nsrc, int L, int cols,
                             void* dst_bf16, int ld_dst, const int* src_lens = nullptr, const int* dst_lens = nullptr);

struct CnnWeights {                // BN-folded, fragment-ordered (see visual_cnn.cu)
  const uint32_t* w1; const float* b1;
  const uint32_t* w2; const float* b2;
  const uint32_t* w3; const float* b3;
  const uint32_t *w1l, *w2l, *w3l;   // lo parts (fp32-grade split path), fragment-ordered like w1/w2/w3
};
// frames (M,H,W) fp32 -> pooled (M,128) operand precision.  frame_lens (variable-length batch of N-frame utterances, or
// null): frames past an utterance's length are not read and go through the network as zero frames.
const char* launch_visual_cnn(cudaStream_t s, int prec, const float* frames, int M, int H, int W, const CnnWeights& w,
                              void* pooled, int num_sms, const int* frame_lens = nullptr, int N = 1);
// tcgen05 fast path for 32x32 frames, bf16 (visual_cnn_tc.cu)
size_t visual_cnn_tc_w2_bytes();
size_t visual_cnn_tc_w3_bytes();
void visual_cnn_tc_pack(const float* w2, const float* w3, uint8_t* w2_slabs, uint8_t* w3_rows);
const char* launch_visual_cnn_tc(LaunchCtx lc, const float* frames, int M, const CnnWeights& w, const uint8_t* w2_slabs,
                                 const uint8_t* w3_rows, void* pooled, int num_sms,
                                 unsigned long long* trace = nullptr, const int* frame_lens = nullptr, int N = 1);
size_t visual_cnn_pack_sizes(int which);   // elements of packed w1/w2/w3 (uint32)
void visual_cnn_pack(const float* w1, const float* w2, const float* w3, uint32_t* p1, uint32_t* p2, uint32_t* p3,
                     bool lo_part = false);

// ---- rows either side of the path (synth.cu) ----
struct SynthProblem {
  int B, S, n, nfft, hop, nf, Hh, Ww;
  double duration;
  const double *amps, *freqs, *phases;   // (B,S)
  const float* noise;                    // (B,S,nf,ph,pw) or null
  float* waves;                          // scratch (B, S+1, n)
  float *mixed_spec, *lip_frames, *clean_specs;
};
// A batch is three launches: launch_synth_waves checks the whole problem and writes the (B, S+1, n) signals, the
// mixture first; launch_stft in the synthesis layout turns them into mixed_spec and clean_specs; launch_synth_lips draws
// the lip frames from them.
const char* launch_synth_waves(cudaStream_t s, const SynthProblem& p);
const char* launch_synth_lips(cudaStream_t s, const SynthProblem& p);
const char* launch_eval_snr(cudaStream_t s, const float* separated, const float* targets, const float* mixed, int B,
                            int S, int FT, double* input_snr, double* output_snr, int* best_perm, double* si_snr);

// ---- waveform side (waveform.cu): STFT analysis with the reference's framing, masked inverse STFT ----
bool fft_size_ok(int nfft);               // a power of two in [8, 2048]: the sizes the transforms take
bool fft_geometry_ok(int nfft, int hop);  // fft_size_ok and 1 <= hop <= nfft: frames that leave no sample out
const char* fft512_init_tables();   // window + twiddle tables of the n_fft = 512 kernels, once per device (avsep_create)
// STFT analysis of signals of L samples: T = 1 + L / hop frames, F = nfft / 2 + 1 bins; a radix-8 register transform for
// nfft = 512, a shared-memory radix-2 one otherwise.  The caller checks fft_size_ok(nfft), hop >= 1 and B, L >= 1.
//   S1 = 0: waves (B, L) -> spec (B, F, T) complex64 and mag (B, F, T) float, either may be null.  lengths: device
//           int32 [B] samples per utterance, or null (all L); the variable-length kernel runs when lengths or
//           frame_lengths (device int32 [B], receives 1 + length / hop) is given.
//   S1 > 0: the synthesis layout, waves (B, S1, L) with the mixture as signal 0 -> magnitudes only: mag (B, F, T) of
//           the mixture, mag2 (B, S1 - 1, F, T) of the other signals or null.  spec, lengths, frame_lengths null.
//   xp (S1 = 0 only, or null): also the forward's Conv1d operand, launch_prep_audio's xp [B * (T + 2), Fp] in operand
//           precision xp_prec, bit-identical to launch_prep_audio of mag with the frame_lengths as its lens.
// B * max(S1, 1) above 65535 is "stft: launch failed".
const char* launch_stft(cudaStream_t s, const float* waves, const int* lengths, int B, int S1, int L, int nfft, int hop,
                        float* spec, float* mag, float* mag2, int* frame_lengths, void* xp = nullptr, int Fp = 0,
                        int xp_prec = PREC_BF16);
// lengths as for launch_stft: the istft runs its variable-length kernel when it is given.
const char* launch_istft_masked(cudaStream_t s, const float* spec, const float* masks, const int* lengths, int B, int S,
                                int T, int nfft, int hop, int L, float* waves);

}  // namespace avsep
