// The steps either side of the forward path, resident on the GPU (SURVEY §8f rows 1 and 3):
//
//   input synthesis   SyntheticAVDataset.__getitem__ / _stft / _make_lip_frame  (reference dataset.py:70-151)
//   SNR evaluation    snr_db / _permutation_snr (demo.py:25-29,67-80), si_snr (losses.py:14-42)
//
// The reference draws a handful of random numbers per item from numpy's PCG64 and then spends its time in a Python
// loop of 3 x 63 windowed rFFTs and 50 frame paintings per item.  Here the draws stay on the host (they are inputs:
// amplitudes, jittered frequencies, phases, patch noise) and the arithmetic runs on the device: fp64 waveform
// synthesis rounded to fp32 exactly where the reference rounds; the STFT of waveform.cu's analysis kernels (launch_stft:
// Hann window in fp64, fp32 FFT like numpy's single-precision pocketfft), magnitudes written in the (B, F, T) layout
// the forward consumes; frame energies by block reduction; patches painted with the clip.  All HBM-bound /
// latency-bound CUDA-core work: no tensor cores.
#include "common.cuh"
#include "kernels.h"

namespace avsep {

namespace {

constexpr double kPi = 3.141592653589793238462643383279502884;

// clean[b,s,i] = float(amp * sin(((2*pi)*f) * t_i + phase)), t_i = i * (duration / n)   (dataset.py:60,78-83)
// mixed[b,i]   = fp32 sum over speakers in speaker order                                  (dataset.py:85)
// waves layout: (B, S+1, n) with the mixture as signal 0 and speaker s as signal 1+s.
__global__ void synth_wave_kernel(const double* __restrict__ amps, const double* __restrict__ freqs,
                                  const double* __restrict__ phases, int S, int n, double step,
                                  float* __restrict__ waves) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double t = __dmul_rn(static_cast<double>(i), step);
  float mix = 0.f;
  for (int s = 0; s < S; ++s) {
    const double c = __dmul_rn(__dmul_rn(2.0, kPi), freqs[b * S + s]);
    const double arg = __dadd_rn(__dmul_rn(c, t), phases[b * S + s]);
    const float x = static_cast<float>(__dmul_rn(amps[b * S + s], sin(arg)));
    waves[(static_cast<size_t>(b) * (S + 1) + 1 + s) * n + i] = x;
    mix = __fadd_rn(mix, x);
  }
  waves[static_cast<size_t>(b) * (S + 1) * n + i] = mix;
}

// One warp per (b, speaker, video frame), no block-level synchronisation: energy = fp32 mean of x^2 over the frame's
// audio span, brightness = min(1, 20*energy), patch = clip(float(brightness) + noise, 0, 1) in the centre 50 %, zeros
// elsewhere (dataset.py:91-104,137-147).
__global__ void __launch_bounds__(256) lip_frames_kernel(const float* __restrict__ waves,
                                                         const float* __restrict__ noise, int B, int S, int n, int nf,
                                                         int Hh, int Ww, float* __restrict__ frames) {
  const long long wid = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (wid >= static_cast<long long>(B) * S * nf) return;
  const int lane = threadIdx.x & 31;
  const int fi = static_cast<int>(wid % nf);
  const long long bs = wid / nf;                 // b * S + s
  const int s = static_cast<int>(bs % S), b = static_cast<int>(bs / S);
  const int step = n / nf;
  const int a = fi * step;
  const int e = min(a + step, n);
  const float* x = waves + (static_cast<size_t>(b) * (S + 1) + 1 + s) * n;
  float acc = 0.f;
  for (int i = a + lane; i < e; i += 32) acc = fmaf(x[i], x[i], acc);
  acc = warp_sum(acc);
  const float energy = acc / static_cast<float>(e - a);
  const float bright = static_cast<float>(fmin(1.0, static_cast<double>(energy) * 20.0));
  const int h0 = Hh / 4, h1 = 3 * Hh / 4, w0 = Ww / 4, w1 = 3 * Ww / 4;
  const int ph = h1 - h0, pw = w1 - w0;
  float* out = frames + static_cast<size_t>(wid) * Hh * Ww;
  const float* nz = noise ? noise + static_cast<size_t>(wid) * ph * pw : nullptr;
  for (int p = lane; p < Hh * Ww; p += 32) {
    const int y = p / Ww, xq = p - y * Ww;
    float v = 0.f;
    if (y >= h0 && y < h1 && xq >= w0 && xq < w1) {
      const float nv = nz ? nz[(y - h0) * pw + (xq - w0)] : 0.f;
      v = fminf(fmaxf(__fadd_rn(bright, nv), 0.f), 1.0f);
    }
    out[p] = v;
  }
}

// ---- SNR evaluation ---------------------------------------------------------------------------------------------
// One CTA per utterance.  Sums (fp64 accumulation of fp32 products):
//   tt[t] = sum tg_t^2, in[t] = sum (mixed - tg_t)^2, d[s][t] = sum (sep_s - tg_t)^2,
//   and for si_snr over the flattened (S,F,T) row: se, st, see, stt, set.
constexpr int MAXS = 4;

__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double r = 0.0;
  for (int i = 0; i < (blockDim.x >> 5); ++i) r += red[i];
  return r;
}

__device__ __forceinline__ double snr_db_f32(double sig_sum, double noise_sum, double count) {
  // demo.py:25-29 with float32 means: sig/(noise + eps) + eps evaluated in float32, log10 in double
  const float sp = static_cast<float>(sig_sum / count);
  const float np_ = static_cast<float>(noise_sum / count);
  const float ratio = __fadd_rn(__fdiv_rn(sp, __fadd_rn(np_, 1e-8f)), 1e-8f);
  return 10.0 * log10(static_cast<double>(ratio));
}

__global__ void eval_snr_kernel(const float* __restrict__ separated, const float* __restrict__ targets,
                                const float* __restrict__ mixed, int S, int FT, double* __restrict__ input_snr,
                                double* __restrict__ output_snr, int* __restrict__ best_perm,
                                double* __restrict__ si_snr) {
  __shared__ double red[32];
  __shared__ double s_d[MAXS * MAXS], s_tt[MAXS], s_in[MAXS];
  const int b = blockIdx.x;
  const float* sep = separated + static_cast<size_t>(b) * S * FT;
  const float* tg = targets + static_cast<size_t>(b) * S * FT;
  const float* mx = mixed ? mixed + static_cast<size_t>(b) * FT : nullptr;
  double d[MAXS * MAXS], tt[MAXS], in[MAXS];
  double se = 0, st = 0, see = 0, stt = 0, set = 0;
#pragma unroll
  for (int i = 0; i < MAXS * MAXS; ++i) d[i] = 0;
#pragma unroll
  for (int i = 0; i < MAXS; ++i) tt[i] = in[i] = 0;
  for (int i = threadIdx.x; i < FT; i += blockDim.x) {
    float tv[MAXS], sv[MAXS];
#pragma unroll
    for (int s = 0; s < MAXS; ++s) {
      tv[s] = s < S ? tg[static_cast<size_t>(s) * FT + i] : 0.f;
      sv[s] = s < S ? sep[static_cast<size_t>(s) * FT + i] : 0.f;
    }
    const float m = mx ? mx[i] : 0.f;
#pragma unroll
    for (int t = 0; t < MAXS; ++t) {
      if (t < S) {
        tt[t] += static_cast<double>(tv[t] * tv[t]);
        const float dm = m - tv[t];
        in[t] += static_cast<double>(dm * dm);
        se += sv[t]; st += tv[t];
        see += static_cast<double>(sv[t]) * sv[t]; stt += static_cast<double>(tv[t]) * tv[t];
        set += static_cast<double>(sv[t]) * tv[t];
#pragma unroll
        for (int s = 0; s < MAXS; ++s) {
          if (s < S) {
            const float df = sv[s] - tv[t];
            d[s * MAXS + t] += static_cast<double>(df * df);
          }
        }
      }
    }
  }
  for (int t = 0; t < S; ++t) {
    const double a = block_sum(tt[t], red), c = block_sum(in[t], red);
    if (threadIdx.x == 0) { s_tt[t] = a; s_in[t] = c; }
    for (int s = 0; s < S; ++s) {
      const double v = block_sum(d[s * MAXS + t], red);
      if (threadIdx.x == 0) s_d[s * MAXS + t] = v;
    }
  }
  se = block_sum(se, red); st = block_sum(st, red); see = block_sum(see, red); stt = block_sum(stt, red);
  set = block_sum(set, red);
  __syncthreads();
  if (threadIdx.x != 0) return;
  const double cnt = static_cast<double>(FT);
  if (input_snr && mx)
    for (int t = 0; t < S; ++t) input_snr[b * S + t] = snr_db_f32(s_tt[t], s_in[t], cnt);       // demo.py:55-58
  // best permutation (demo.py:67-80): separated[perm[t]] is matched with targets[t]
  double snr[MAXS * MAXS];
  for (int s = 0; s < S; ++s)
    for (int t = 0; t < S; ++t) snr[s * MAXS + t] = snr_db_f32(s_tt[t], s_d[s * MAXS + t], cnt);
  int perm[MAXS] = {0, 1, 2, 3}, bestp = 0, code = 0;
  double best = -1e9;
  // iterate permutations of S items in lexicographic order (itertools.permutations order)
  int nperm = 1;
  for (int i = 2; i <= S; ++i) nperm *= i;
  for (int pi = 0; pi < nperm; ++pi) {
    // decode the pi-th lexicographic permutation (factorial number system)
    int avail[MAXS] = {0, 1, 2, 3};
    int rem = pi, fact = nperm;
    for (int pos = 0; pos < S; ++pos) {
      fact /= (S - pos);
      const int k = rem / fact;
      rem -= k * fact;
      perm[pos] = avail[k];
      for (int q = k; q < S - 1 - pos; ++q) avail[q] = avail[q + 1];
    }
    double sum = 0;
    code = 0;
    for (int t = 0; t < S; ++t) { sum += snr[perm[t] * MAXS + t]; code = code * MAXS + perm[t]; }
    const double val = sum / S;
    if (val > best) { best = val; bestp = code; }
  }
  if (output_snr) output_snr[b] = best;
  if (best_perm) best_perm[b] = bestp;
  if (si_snr) {                                                                                  // losses.py:14-42
    const double nn = static_cast<double>(S) * FT;
    const double me = se / nn, mt = st / nn;
    const double dot = set - nn * me * mt;
    const double e_t = stt - nn * mt * mt;
    const double e_e = see - nn * me * me;
    const double alpha = dot / (e_t + 1e-8);
    const double pp = alpha * alpha * e_t;
    const double nz = e_e - 2.0 * alpha * dot + alpha * alpha * e_t;
    si_snr[b] = 10.0 * log10(pp / (fmax(nz, 0.0) + 1e-8) + 1e-8);
  }
}

}  // namespace

const char* launch_synth_waves(cudaStream_t s, const SynthProblem& p) {
  if (p.B <= 0) return "synth: empty batch";
  if (p.S < 1 || p.S > 8) return "synth: num_speakers must be 1..8";
  if (!fft_size_ok(p.nfft)) return "synth: n_fft must be a power of two in [8, 2048]";
  if (p.n < 1 || p.hop < 1 || p.nf < 1 || p.Hh < 1 || p.Ww < 1) return "synth: bad geometry";
  if (p.nf > p.n) return "synth: more video frames than audio samples";
  if (static_cast<long long>(p.B) * (p.S + 1) > 65535) return "synth: batch * (speakers + 1) above 65535";
  synth_wave_kernel<<<dim3((p.n + 255) / 256, p.B), 256, 0, s>>>(p.amps, p.freqs, p.phases, p.S, p.n,
                                                                 p.duration / static_cast<double>(p.n), p.waves);
  return cudaGetLastError() == cudaSuccess ? nullptr : "synth: launch failed";
}

const char* launch_synth_lips(cudaStream_t s, const SynthProblem& p) {
  const long long lip_warps = static_cast<long long>(p.B) * p.S * p.nf;
  lip_frames_kernel<<<static_cast<unsigned>((lip_warps + 7) / 8), 256, 0, s>>>(p.waves, p.noise, p.B, p.S, p.n, p.nf,
                                                                              p.Hh, p.Ww, p.lip_frames);
  return cudaGetLastError() == cudaSuccess ? nullptr : "synth: launch failed";
}

const char* launch_eval_snr(cudaStream_t s, const float* separated, const float* targets, const float* mixed, int B,
                            int S, int FT, double* input_snr, double* output_snr, int* best_perm, double* si_snr) {
  if (B <= 0 || FT <= 0) return "eval_snr: empty problem";
  if (S < 1 || S > MAXS) return "eval_snr: num_speakers must be 1..4";
  eval_snr_kernel<<<B, 512, 0, s>>>(separated, targets, mixed, S, FT, input_snr, output_snr, best_perm, si_snr);
  return cudaGetLastError() == cudaSuccess ? nullptr : "eval_snr: launch failed";
}

}  // namespace avsep
