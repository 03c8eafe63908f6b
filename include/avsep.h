/*
 * avsep.h - C ABI of the B200-native AVSeparationTransformer forward path (libavsep.so).
 *
 * The reference (danieleschmidt/AV-Separation-Transformer) is pure Python on PyTorch and has no
 * FFI / operator / plugin layer of its own: its drop-in boundary for this path is the nn.Module
 *     AVSeparationTransformer.__init__(freq_bins, d_model, nhead, num_encoder_layers,
 *                                      num_fusion_layers, num_speakers, dropout)      model.py:240-249
 *     AVSeparationTransformer.forward(mixed_spec, lip_frames) -> (separated, masks)    model.py:268-276
 * plus its state_dict key set (SURVEY.md Appendix A).  The entry points below are what a ctypes/pybind
 * binding of that module binds instead of torch.nn: plain pointers and sizes, no torch types.
 * INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; avsep_last_error(h) gives the message.
 *     No C++ exception crosses this boundary.
 *   - a handle is bound to one CUDA device; calls are stream-ordered on the caller's stream and never
 *     synchronise internally (except avsep_forward_host and the *_debug / *_test helpers).
 *   - device buffers are owned by the caller; the library owns only the prepacked weights and, when the
 *     caller passes workspace == NULL, a cached workspace per shape.
 *   - eval-mode semantics only (dropout = identity, BatchNorm running statistics): model.py:159,164,197,288.
 */
#ifndef AVSEP_H_
#define AVSEP_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define AVSEP_API __attribute__((visibility("default")))
#else
#define AVSEP_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct avsep_handle avsep_handle;

enum { AVSEP_PREC_BF16 = 0, AVSEP_PREC_TF32 = 1 };
enum { AVSEP_DTYPE_F32 = 0, AVSEP_DTYPE_I64 = 1 };

/* Constructor arguments of the reference module (model.py:240-249) + execution options. */
typedef struct avsep_config {
  int32_t freq_bins;
  int32_t d_model;
  int32_t nhead;
  int32_t num_encoder_layers;
  int32_t num_fusion_layers;
  int32_t num_speakers;
  int32_t precision; /* AVSEP_PREC_*: operand precision of the tensor-core contractions */
  int32_t device;    /* CUDA device ordinal */
} avsep_config;

/* Replaces AVSeparationTransformer.__init__ (model.py:240-266). */
AVSEP_API int avsep_create(const avsep_config* cfg, avsep_handle** out);
AVSEP_API void avsep_destroy(avsep_handle* h);
AVSEP_API const char* avsep_last_error(const avsep_handle* h); /* h may be NULL: error of the last failed create */

/* Replaces nn.Module.load_state_dict: one call per state_dict entry, reference key names
 * (SURVEY.md Appendix A, e.g. "audio_encoder.input_proj.0.weight"), HOST pointer, fp32 (or int64 for
 * num_batches_tracked, which is accepted and ignored).  Data is copied. */
AVSEP_API int avsep_set_weight(avsep_handle* h, const char* key, const void* host_data, int32_t dtype, const int64_t* shape,
                     int32_t ndim);
/* BN fold, Conv1d tap repack, operand-precision cast, upload.  Fails if a key is missing or mis-shaped. */
AVSEP_API int avsep_finalize_weights(avsep_handle* h, void* cuda_stream);

/* Scratch bytes avsep_forward needs for this shape (0 on error). */
AVSEP_API size_t avsep_workspace_bytes(avsep_handle* h, int32_t B, int32_t T, int32_t N, int32_t Hh, int32_t Ww);

/* Replaces AVSeparationTransformer.forward (model.py:268-276).  DEVICE pointers:
 *   mixed_spec (B,F,T) fp32, lip_frames (B,N,Hh,Ww) fp32 -> separated, masks (B,S,F,T) fp32 contiguous.
 * workspace may be NULL (library-owned, cached per shape). */
AVSEP_API int avsep_forward(avsep_handle* h, const float* mixed_spec, const float* lip_frames, int32_t B, int32_t T, int32_t N,
                  int32_t Hh, int32_t Ww, float* separated, float* masks, void* workspace, size_t workspace_bytes,
                  void* cuda_stream);

/* Variable-length batch.  mixed_spec (B,F,T), lip_frames (B,N,Hh,Ww) hold each utterance left-aligned in the
 * first lengths[b] frames / frame_lengths[b] lip frames; T and N are the batch maxima.  lengths, frame_lengths:
 * DEVICE int32 [B], or NULL for "all T" / "all N".  For each b the outputs [b, :, :, :lengths[b]] equal the
 * outputs of avsep_forward on that utterance alone at (lengths[b], frame_lengths[b]); [b, :, :, lengths[b]:] are 0
 * in both separated and masks.  Input values past the lengths are never read (NaN there is harmless).
 * Lengths are read on the device (no host sync; a captured graph replays with whatever the buffers hold then);
 * values outside [1, T] / [1, N] behave as the nearest bound.  Workspace: avsep_workspace_bytes(B, T, N, Hh, Ww). */
AVSEP_API int avsep_forward_varlen(avsep_handle* h, const float* mixed_spec, const float* lip_frames,
                                   const int32_t* lengths, const int32_t* frame_lengths, int32_t B, int32_t T,
                                   int32_t N, int32_t Hh, int32_t Ww, float* separated, float* masks,
                                   void* workspace, size_t workspace_bytes, void* cuda_stream);

/* Same call with HOST buffers (pinned memory recommended): H2D copies, forward and D2H copies are issued on
 * the stream and the call returns after the results have landed (the e2e path of bench.py). */
AVSEP_API int avsep_forward_host(avsep_handle* h, const float* mixed_spec, const float* lip_frames, int32_t B, int32_t T,
                       int32_t N, int32_t Hh, int32_t Ww, float* separated, float* masks, void* cuda_stream);

/* Streaming form of avsep_forward_host for back-to-back batches (the demo.py:45-50 loop over a dataset): enqueues the
 * copy-in / kernels / copy-out pipeline of one batch on I/O slot 0 .. AVSEP_HOST_SLOTS - 1 and returns;
 * avsep_host_wait(slot) returns when that slot's results are in the host buffers.  Cycling through the slots overlaps
 * the copy-in of batch i+1 with the kernels and copy-out of batch i (two slots are enough for that; a third keeps both
 * PCIe directions busy across the hand-over).  Host buffers must be pinned for the copies to be asynchronous, and must stay
 * valid (inputs) / untouched (outputs) until the wait.  A slot is reused only after its previous batch has finished
 * with its device buffers (ordered on the device; the caller only has to wait before reading results). */
#define AVSEP_HOST_SLOTS 4
AVSEP_API int avsep_forward_host_async(avsep_handle* h, const float* mixed_spec, const float* lip_frames, int32_t B,
                                       int32_t T, int32_t N, int32_t Hh, int32_t Ww, float* separated, float* masks,
                                       int32_t slot, void* cuda_stream);
AVSEP_API int avsep_host_wait(avsep_handle* h, int32_t slot);

/* Number of kernels the last avsep_forward on this handle launched. */
AVSEP_API int64_t avsep_last_launch_count(const avsep_handle* h);

/* Sub-module forwards (reference: AudioEncoder.forward model.py:54-60, VisualEncoder.forward model.py:103-117,
 * CrossModalFusion.forward model.py:145-149, SeparationDecoder.forward/.separate model.py:201-220).
 * DEVICE pointers, fp32, contiguous. */
AVSEP_API int avsep_audio_encoder(avsep_handle* h, const float* mixed_spec, int32_t B, int32_t T, float* out_BTd,
                        void* cuda_stream);
AVSEP_API int avsep_visual_encoder(avsep_handle* h, const float* lip_frames, int32_t B, int32_t N, int32_t Hh, int32_t Ww,
                         int32_t target_len, float* out_BTd, void* cuda_stream);
AVSEP_API int avsep_fusion(avsep_handle* h, const float* audio_BTd, const float* visual_BLd, int32_t B, int32_t T, int32_t L,
                 float* out_BTd, void* cuda_stream);
AVSEP_API int avsep_decoder(avsep_handle* h, const float* fused_BTd, const float* mixed_spec, int32_t B, int32_t T,
                  float* separated, float* masks, void* cuda_stream);

/* Debug: when enabled, avsep_forward keeps fp32 snapshots of intermediate stages
 * ("audio_embed", "audio_enc", "visual_pool", "visual_embed", "visual_enc", "fused"). */
AVSEP_API int avsep_set_debug(avsep_handle* h, int32_t enable);
/* Copies a snapshot to a HOST buffer of `capacity` floats; returns the element count in *count. Synchronises. */
AVSEP_API int avsep_debug_get_stage(avsep_handle* h, const char* name, float* host_out, size_t capacity, size_t* count);

/* Execution options.  Apart from them, kernel choice follows from the configuration, the shapes and debug mode alone.
 * name -> meaning (default):
 *   "use_graph" (1)          CUDA-graph replay keyed by (shape, buffers)
 *   "two_stream" (1)         audio and visual branches on two streams
 *   "pdl" (1)                programmatic dependent launch between consecutive kernels
 *   "attn_tc" (1)            1: tcgen05 attention when usable and min(Lq, Lk) >= 96; 0: never; 2: whenever usable
 *   "host_chunk" (0), "host_lanes" (0)    host-buffer pipeline: utterances per chunk, concurrent compute lanes; 0 = auto
 *                            (56 x 2 lanes for avsep_forward_host, 128 x 1 lane for avsep_forward_host_async)
 *   "profile_spin_us"        length of the GPU spin kernel that precedes a profiled forward
 * Any other name is an error.  The environment variable AVSEP_OPTS="name=value,name=value" applies options at
 * avsep_create (measurement runs).  "pdl" is process-wide: it applies to every handle of the process, not only to `h`;
 * every other option applies to `h` alone. */
AVSEP_API int avsep_set_option(avsep_handle* h, const char* name, int32_t value);

/* Per-kernel timing: when enabled every launch of the forward is bracketed by a cudaEvent pair on the launching
 * stream.  avsep_profile_report synchronises and writes one "label launches total_ms" line per kernel class. */
AVSEP_API int avsep_set_profile(avsep_handle* h, int32_t enable);
AVSEP_API int avsep_profile_report(avsep_handle* h, char* buf, size_t capacity, int32_t reset);

/* Kernel-level test hooks (DEVICE pointers; used by tests/ to check each kernel against a torch fp32 reference).
 *   gemm: out[M,N] = act(A[M,K] @ W[N,K]^T + bias), A/W in operand precision (bf16 or fp32), out fp32.
 *   gemm_ln: x += A W^T + bias (fp32, in place); out_op = LayerNorm(x) -- the fused sub-layer epilogue.
 *   ffn_fused: x += W2 act(W1 a + b1) + b2 (fp32, in place); out_op = LayerNorm(x); d_model = 256, bf16 only.
 *   conv1d: taps=3 implicit GEMM over a zero-haloed activation: A [B*(L+2), K], W [N, 3*K] (k = tap*K + c),
 *           out fp32 [B*L, N] (ROW_PAD2COMPACT).
 *   attention: q [B*Lq, H*hd], k/v [B*Lk, H*hd] bf16 (lerp_src = 0) or fp32 [B*lerp_src, H*hd] (lerp on load).
 *   add_layernorm: x_out = x + y, out = LN(x_out) in operand precision.
 *   visual_cnn: frames (M,Hh,Ww) -> pooled (M,128) operand precision, using the handle's conv weights. */
AVSEP_API int avsep_test_gemm(avsep_handle* h, const void* A, const void* W, const float* bias, float* out, int32_t M, int32_t N,
                    int32_t K, int32_t act, int32_t force_bn, void* cuda_stream);
AVSEP_API int avsep_test_gemm_ln(avsep_handle* h, const void* A, const void* W, const float* bias, float* x_inout,
                                 const float* gamma, const float* beta, void* out_op, int32_t M, int32_t N, int32_t K,
                                 void* cuda_stream);
AVSEP_API int avsep_test_gemm_trace(avsep_handle* h, const void* A, const void* W, const float* bias, float* x_or_out,
                                    const float* gamma, const float* beta, void* out_op, int32_t M, int32_t N, int32_t K,
                                    int32_t ln, int32_t act, unsigned long long* trace_dev, void* cuda_stream);
AVSEP_API int avsep_test_ffn_fused(avsep_handle* h, const void* a, const void* w1, const float* b1, const void* w2,
                                   const float* b2, int32_t act, float* x_inout, const float* gamma, const float* beta,
                                   void* out_op, int32_t M, void* cuda_stream);
AVSEP_API int avsep_test_ffn_fused_trace(avsep_handle* h, const void* a, const void* w1, const float* b1, const void* w2,
                                         const float* b2, int32_t act, float* x_inout, const float* gamma,
                                         const float* beta, void* out_op, int32_t M, unsigned long long* trace_dev,
                                         void* cuda_stream);
AVSEP_API int avsep_test_conv1d(avsep_handle* h, const void* A_padded, const void* W3, const float* bias, float* out, int32_t B,
                      int32_t L, int32_t N, int32_t K, void* cuda_stream);
AVSEP_API int avsep_test_attention(avsep_handle* h, const void* q, const void* k, const void* v, void* out, int32_t B, int32_t H,
                         int32_t hd, int32_t Lq, int32_t Lk, int32_t lerp_src, void* cuda_stream);
AVSEP_API int avsep_test_add_layernorm(avsep_handle* h, const float* x, const float* y, const float* gamma, const float* beta,
                             float* x_out, void* out_op, int32_t M, int32_t d, void* cuda_stream);
AVSEP_API int avsep_test_visual_cnn(avsep_handle* h, const float* frames, int32_t M, int32_t Hh, int32_t Ww, void* pooled,
                          void* cuda_stream);
AVSEP_API int avsep_test_visual_cnn_trace(avsep_handle* h, const float* frames, int32_t M, void* pooled,
                                          unsigned long long* trace_dev, void* cuda_stream);

/* ---------------------------------------------------------------------------------------------------------------
 * The rows either side of the path (SURVEY.md section 8f, ranks 1 and 3).  All pointers are DEVICE pointers.
 * ------------------------------------------------------------------------------------------------------------- */

/* Geometry of the reference's SyntheticAVDataset (reference src/av_separation/dataset.py:33-65). */
typedef struct avsep_synth_config {
  int32_t num_samples_audio;  /* int(sample_rate * duration), dataset.py:59 */
  double duration;            /* seconds (t = linspace(0, duration, n, endpoint=False), dataset.py:60) */
  int32_t n_fft;              /* power of two, <= 2048; freq_bins = n_fft/2 + 1 */
  int32_t hop_length;         /* T = 1 + num_samples_audio / hop_length, dataset.py:65 */
  int32_t num_frames;         /* video frames per speaker; the item holds num_speakers * num_frames frames */
  int32_t frame_h, frame_w;
  int32_t num_speakers;
} avsep_synth_config;

/* Replaces SyntheticAVDataset.__getitem__ for a batch (dataset.py:70-119, _stft :122-135, _make_lip_frame :137-147).
 * The reference's random draws are inputs (consume numpy's default_rng(idx) in the reference's order on the host):
 *   amps, freqs (already jittered), phases : (B, S) float64;  noise : (B, S, num_frames, H/2-ish, W/2-ish) float32
 *   patch noise N(0, 0.05), or NULL for none.
 * Outputs: mixed_spec (B, F, T), lip_frames (B, S*num_frames, H, W), clean_specs (B, S, F, T) or NULL, float32. */
AVSEP_API int avsep_synth_batch(avsep_handle* h, const avsep_synth_config* cfg, int32_t B, const double* amps,
                                const double* freqs, const double* phases, const float* noise, float* mixed_spec,
                                float* lip_frames, float* clean_specs, void* cuda_stream);

/* Replaces the per-utterance SNR evaluation after the path: snr_db / _permutation_snr of evaluate_separation
 * (reference demo.py:25-29,55-62,67-80) and the per-row value of si_snr (src/av_separation/losses.py:14-42).
 *   separated, targets : (B, S, F, T) float32;  mixed : (B, F, T) float32 or NULL
 * Outputs (any may be NULL): input_snr (B, S) float64 dB; output_snr (B) float64 dB = best-permutation mean;
 * best_perm (B) int32 = the chosen permutation as base-4 digits (digit t = index of the separated channel matched
 * with target t, most significant first); si_snr (B) float64 dB over the flattened (S, F, T) row.  S <= 4. */
AVSEP_API int avsep_eval_snr(avsep_handle* h, const float* separated, const float* targets, const float* mixed,
                             int32_t B, int32_t S, int32_t F, int32_t T, double* input_snr, double* output_snr,
                             int32_t* best_perm, double* si_snr, void* cuda_stream);

/* ---------------------------------------------------------------------------------------------------------------
 * The waveform side (SURVEY.md section 8f, rank 4).  The reference has no counterpart: it works on magnitude
 * spectrograms only and lists "STFT phase / iSTFT reconstruction" as missing (reference README.md:140).  The
 * analysis keeps the framing of SyntheticAVDataset._stft (dataset.py:122-135): frame i starts at i*hop_length (no
 * centring), is zero-padded past the end of the signal and weighted by np.hanning(n_fft); T = 1 + L / hop_length.
 * ------------------------------------------------------------------------------------------------------------- */

/* waves (B, L) float32 -> spec (B, F, T) complex64 (interleaved re, im), F = n_fft/2 + 1; mag (B, F, T) float32 or
 * NULL receives |spec|, bit-identical to the mixed_spec avsep_synth_batch produces from the same samples. */
AVSEP_API int avsep_stft(avsep_handle* h, const float* waves, int32_t B, int32_t L, int32_t n_fft, int32_t hop_length,
                         float* spec, float* mag, void* cuda_stream);

/* Masked inverse: waves[b,s,n] = sum_i w[n-i*hop] * irfft(masks[b,s,:,i] * spec[b,:,i])[n-i*hop] / sum_i w^2[n-i*hop]
 * (weighted overlap-add; numpy irfft semantics; samples with a zero window sum - n = 0 - are 0).
 *   spec (B, F, T) complex64; masks (B, S, F, T) float32, or NULL with S = 1 for the plain inverse;
 *   waves (B, S, L) float32 with L <= (T-1)*hop_length + n_fft.  avsep_istft(avsep_stft(x)) == x for n >= 1. */
AVSEP_API int avsep_istft(avsep_handle* h, const float* spec, const float* masks, int32_t B, int32_t S, int32_t T,
                          int32_t n_fft, int32_t hop_length, int32_t L, float* waves, void* cuda_stream);

/* Variable-length waveform batches (the waveform counterpart of avsep_forward_varlen).  Utterance b sits
 * left-aligned in its padded row and owns its first L_b = lengths[b] samples; lengths is a DEVICE int32 [B] array in
 * samples, read on the device only (no host sync; a captured graph replays with whatever it holds then), values
 * outside [1, L] behave as the nearest bound, and NULL means "all L" (avsep_stft / avsep_istft are these calls with
 * NULL lengths).  Geometry, checks and errors are those of avsep_stft / avsep_istft; each call is one kernel launch.
 *   avsep_stft_varlen: T = 1 + L / hop_length is the batch's frame count and T_b = 1 + L_b / hop_length the
 *     utterance's.  spec / mag [b, :, :T_b] equal avsep_stft of waves[b, :L_b] alone, bit for bit; [b, :, T_b:] are
 *     0; samples past L_b are never read.  frame_lengths_out: DEVICE int32 [B] receiving T_b (exactly the `lengths`
 *     argument avsep_forward_varlen takes), or NULL.  With NULL lengths and non-NULL frame_lengths_out every entry is T.
 *   avsep_istft_varlen: with T_b = min(T, 1 + L_b / hop_length), waves[b, s, :L_b] equal avsep_istft of
 *     spec[b, :, :T_b] and masks[b, s, :, :T_b] alone at length L_b, bit for bit; waves[b, s, L_b:] are 0; spectrum
 *     and mask columns at or past T_b are never read.
 * Both transforms pack two frames into one complex FFT; frames at or past T_b are staged as zeros, so NaN or Inf in
 * the padding never reaches a valid frame through its pair partner. */
AVSEP_API int avsep_stft_varlen(avsep_handle* h, const float* waves, const int32_t* lengths, int32_t B, int32_t L,
                                int32_t n_fft, int32_t hop_length, float* spec, float* mag,
                                int32_t* frame_lengths_out, void* cuda_stream);
AVSEP_API int avsep_istft_varlen(avsep_handle* h, const float* spec, const float* masks, const int32_t* lengths,
                                 int32_t B, int32_t S, int32_t T, int32_t n_fft, int32_t hop_length, int32_t L,
                                 float* waves, void* cuda_stream);

/* Test hook: one whole transformer stack through the fused kernel (csrc/xformer_stack_sm100.cu) on the handle's
 * weights.  which: 0 = AudioEncoder.transformer (model.py:48-52,59), 1 = VisualEncoder.transformer (model.py:97-101,111),
 * 2 = CrossModalFusion.layers (+ .norm when final_ln) (model.py:145-149,166-173) with kv = bf16 [B*L, Lf*2*d] rows holding
 * every layer's projected K | V.  x_in fp32 [B*L, d]; out_x fp32 / out_op bf16 [B*L, d], either may be NULL. */
AVSEP_API int avsep_test_xformer_stack(avsep_handle* h, int32_t which, const float* x_in, const void* kv, int32_t B,
                                       int32_t L, float* out_x, void* out_op, int32_t final_ln, long long* trace_dev,
                                       void* cuda_stream);   /* trace_dev: NULL or [grid][256] clock stamps (tools/stack_trace.py) */

/* Test hook: CrossModalFusion.layers + .norm followed by SeparationDecoder (model.py:166-173,201-220) in the one fused
 * kernel the forward uses: x_in fp32 [B*L, d], kv as above, mixed (B, F, L) fp32 -> separated / masks (B, S, F, L) fp32. */
AVSEP_API int avsep_test_fusion_decoder(avsep_handle* h, const float* x_in, const void* kv, int32_t B, int32_t L,
                                        const float* mixed, float* separated, float* masks, long long* trace_dev,
                                        void* cuda_stream);

/* ---- batch sharding over the GPUs of one box (SURVEY.md 8e; BASELINE.json north_star: "inputs scattered and
 * separated/masks gathered over NVLink") -------------------------------------------------------------------------
 * The path shards by utterance with no collective inside the model (model.py has no op that mixes batch elements in
 * eval mode), so the only inter-GPU traffic is the scatter of the root's inputs and the gather of the outputs.  One
 * process per GPU: the root allocates its global input / output buffers with avsep_shared_alloc, which also returns a
 * 64-byte inter-process handle (cudaIpcMemHandle_t); every other rank maps them with avsep_shared_open and moves its
 * shard with avsep_copy_async, a stream-ordered copy that the copy engines execute over NVLink / NVSwitch peer
 * memory (no SM is taken from the forward kernels, unlike a collective's send/recv CTAs).
 * Ownership: memory from avsep_shared_alloc is freed with avsep_shared_free by the allocating process, mappings from
 * avsep_shared_open are released with avsep_shared_close; both are also released by avsep_destroy. */
#define AVSEP_IPC_HANDLE_BYTES 64
AVSEP_API int avsep_shared_alloc(avsep_handle* h, size_t bytes, void** dev_ptr,
                                 unsigned char handle_out[AVSEP_IPC_HANDLE_BYTES]);
AVSEP_API int avsep_shared_free(avsep_handle* h, void* dev_ptr);
AVSEP_API int avsep_shared_open(avsep_handle* h, const unsigned char handle[AVSEP_IPC_HANDLE_BYTES], void** dev_ptr);
AVSEP_API int avsep_shared_close(avsep_handle* h, void* dev_ptr);
/* dst / src: any mix of this device's memory, peer memory mapped with avsep_shared_open, or pinned host memory. */
AVSEP_API int avsep_copy_async(avsep_handle* h, void* dst, const void* src, size_t bytes, void* cuda_stream);


/* SeparationDecoder.separate (reference model.py:210-220): separated[b,s,f,t] = masks[b,s,f,t] * mixed_spec[b,f,t],
 * masks / separated (B, S, F, T) fp32 contiguous, mixed_spec (B, F, T) fp32; S and F are the handle's (16-byte
 * accesses when masks and separated share their alignment modulo 16, element-wise otherwise).
 * One fp32 multiply per element: bit-identical to the reference's broadcast product and to the `separated` that
 * avsep_forward's decoder epilogue writes. */
AVSEP_API int avsep_separate(avsep_handle* h, const float* masks, const float* mixed_spec, int32_t B, int32_t T,
                             float* separated, void* cuda_stream);

/* Masks-only gather (SURVEY.md 8e, "gather only masks: the root recomputes separated = masks x mixed, which it already
 * holds"): a rank pushes its masks shard with avsep_copy_async and then raises a ticket -- a 32-bit word in memory
 * from avsep_shared_alloc, its own or a mapped peer's -- with avsep_flag_signal on the same stream; the consumer
 * orders its stream after the ticket with avsep_flag_wait (a one-CTA kernel polling its own memory; no host
 * round trip, no collective) and rebuilds the shard's `separated` with avsep_separate.  Tickets only grow; wait
 * succeeds once every flag >= value.  A flag that does not arrive within timeout_s makes the waiting kernel trap (the
 * next CUDA call on the handle's device fails) instead of hanging the stream.  n <= 16. */
AVSEP_API int avsep_flag_signal(avsep_handle* h, uint32_t* const* flags, int32_t n, uint32_t value, void* cuda_stream);
AVSEP_API int avsep_flag_wait(avsep_handle* h, uint32_t* const* flags, int32_t n, uint32_t value, double timeout_s,
                              void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* AVSEP_H_ */
