// The waveform side of the path (SURVEY §8f row 4): the reference stops at magnitude spectrograms and lists
// "STFT phase / iSTFT reconstruction" as missing (reference README.md:140), so a separated utterance never becomes
// audio there.  These two kernels close that gap on the device with the reference's own analysis framing:
//
//   stft_complex_kernel   the framing of SyntheticAVDataset._stft (dataset.py:122-135: frame i starts at i*hop, no
//                         centring, zero-padded past the end, np.hanning window, rfft) keeping the phase: complex64
//                         (B, F, T); |.| is bit-identical to the magnitudes of synth.cu's stft_mag_kernel.
//   istft_masked_kernel   y[b,s,n] = sum_i w[n-i*hop] * irfft(mask[b,s,:,i] * X[b,:,i])[n-i*hop] / sum_i w^2[n-i*hop]
//                         (weighted overlap-add, the least-squares inverse of that analysis; samples no window
//                         reaches with non-zero weight - n = 0 for a Hann window - come out 0).
//
// One CTA owns a run of consecutive output samples and transforms every frame that overlaps it (no atomics, results
// independent of the launch geometry); two Hermitian spectra share one complex inverse transform (z = A + iB ->
// ifft(z) = a + ib for real a, b).  fp32 shared-memory radix-2 transforms, fp64 window: HBM/latency-bound CUDA-core
// work, no tensor cores.
#include "common.cuh"
#include "fft512.cuh"
#include "kernels.h"

namespace avsep {

namespace {

constexpr double kPi = 3.141592653589793238462643383279502884;
constexpr int TGA = 8;   // analysis frames per CTA

__device__ __forceinline__ void fft_stages(float* re, float* im, const float* twr, const float* twi, int log2n,
                                           int tid) {
  for (int s = 1; s <= log2n; ++s) {
    __syncthreads();
    const int half = 1 << (s - 1);
    const int pos = tid & (half - 1);
    const int i0 = ((tid >> (s - 1)) << s) + pos;
    const int i1 = i0 + half;
    const int tw = pos << (log2n - s);
    const float wr = twr[tw], wi = twi[tw];
    const float xr = re[i1], xi = im[i1];
    const float pr = wr * xr - wi * xi, pi = wr * xi + wi * xr;
    const float ar = re[i0], ai = im[i0];
    re[i0] = ar + pr; im[i0] = ai + pi;
    re[i1] = ar - pr; im[i1] = ai - pi;
  }
  __syncthreads();
}

// np.hanning(M)[k] = 0.5 + 0.5*cos(pi*(1-M+2k)/(M-1)), fp64 (dataset.py:124)
__device__ __forceinline__ double hann(int k, int nfft) {
  return 0.5 + 0.5 * cos(kPi * static_cast<double>(1 - nfft + 2 * k) / static_cast<double>(nfft - 1));
}

// Variable-length batch (VARLEN): utterance b owns the first nb = clamp(lengths[b], 1, n) samples of its row (all n
// when lengths is null) and the first Tb = 1 + nb / hop frames.  Samples at or past nb are never read, frames at or
// past Tb are neither staged nor transformed, and their outputs are stored as 0.  Frames are paired by absolute index
// (t0 + g, t0 + g + 1) whatever T is, so frame Tb - 1 has the partner (or the zero partner) it has in a stand-alone
// call at (nb, Tb): the valid frames are bit-identical to that call.  CTA (0, b) writes Tb to frame_lengths[b].
// The uniform instantiation ignores the two trailing parameters and compiles as before they existed.
__device__ __forceinline__ int clamp_len(const int* lengths, int b, int n) {
  return lengths ? min(max(lengths[b], 1), n) : n;
}

// grid (ceil(T/TGA), B), nfft/2 threads.  spec: (B, F, T) float2; mag: (B, F, T) float or null.
template <bool VARLEN>
__global__ void stft_complex_kernel(const float* __restrict__ waves, int n, int nfft, int log2n, int hop, int T, int F,
                                    float2* __restrict__ spec, float* __restrict__ mag,
                                    const int* __restrict__ lengths, int* __restrict__ frame_lengths) {
  extern __shared__ __align__(16) uint8_t sm_raw[];
  double* win = reinterpret_cast<double*>(sm_raw);          // [nfft]
  float* re = reinterpret_cast<float*>(win + nfft);         // [nfft]
  float* im = re + nfft;                                    // [nfft]
  float* twr = im + nfft;                                   // [nfft/2]
  float* twi = twr + nfft / 2;                              // [nfft/2]
  float2* stage = reinterpret_cast<float2*>(twi + nfft / 2);  // [F][TGA]
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * TGA;
  const int tid = threadIdx.x;
  const float* x = waves + static_cast<size_t>(b) * n;
  const int nb = VARLEN ? clamp_len(lengths, b, n) : n;   // this utterance's samples and frames
  const int Tb = VARLEN ? 1 + nb / hop : T;
  if (VARLEN && frame_lengths && blockIdx.x == 0 && tid == 0) frame_lengths[b] = Tb;
  if (!VARLEN || t0 < Tb) {
    float sv, cv;
    sincospif(-2.0f * static_cast<float>(tid) / static_cast<float>(nfft), &sv, &cv);
    twr[tid] = cv; twi[tid] = sv;
    win[tid] = hann(tid, nfft);
    win[tid + nfft / 2] = hann(tid + nfft / 2, nfft);
  }
  const int ng = min(TGA, Tb - t0);
  for (int g = 0; g < ng; g += 2) {
    const int ta = t0 + g;
    const bool has_b = g + 1 < ng;
    __syncthreads();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int k = tid + h * (nfft / 2);
      const int sa = ta * hop + k, sb = sa + hop;
      const float va = sa < nb ? x[sa] : 0.f;
      const float vb = (has_b && sb < nb) ? x[sb] : 0.f;
      const double w = win[k];
      const int r = static_cast<int>(__brev(static_cast<unsigned>(k)) >> (32 - log2n));
      re[r] = static_cast<float>(static_cast<double>(va) * w);     // float32 `frame *= window`, dataset.py:131
      im[r] = static_cast<float>(static_cast<double>(vb) * w);
    }
    fft_stages(re, im, twr, twi, log2n, tid);
    for (int f = tid; f < F; f += blockDim.x) {
      const int fn = (nfft - f) & (nfft - 1);
      const float zr = re[f], zi = im[f], yr = re[fn], yi = im[fn];
      stage[f * TGA + g] = make_float2(0.5f * (zr + yr), 0.5f * (zi - yi));                 // A = (Z + conj Z~)/2
      if (has_b) stage[f * TGA + g + 1] = make_float2(0.5f * (zi + yi), 0.5f * (yr - zr));  // B = (Z - conj Z~)/2i
    }
  }
  __syncthreads();
  for (int e = tid; e < F * TGA; e += blockDim.x) {
    const int f = e / TGA, g = e - f * TGA;
    if (g >= (VARLEN ? T - t0 : ng)) continue;
    const size_t o = (static_cast<size_t>(b) * F + f) * T + t0 + g;
    const float2 v = (!VARLEN || g < ng) ? stage[e] : make_float2(0.f, 0.f);
    spec[o] = v;
    // same expression as stft_mag_kernel (0.5 * hypot of the unscaled sums) so the magnitudes agree bit for bit
    if (mag) mag[o] = 0.5f * hypotf(2.0f * v.x, 2.0f * v.y);
  }
}

// grid (ceil(L/CH), S, B), nfft/2 threads.  spec (B, F, T) float2, masks (B, S, F, T) float or null (S = 1),
// out (B, S, L).  CH = samples per CTA (a multiple of hop).  The frames that overlap the CTA's samples are processed
// in batches of NB: the masked half spectra of a batch are staged in shared memory with row-contiguous loads (the
// (F, T) layout puts the frames of one bin side by side, so a per-frame gather would touch one sector per element),
// then transformed two at a time.
constexpr int NB = 12;        // frames per staged batch (even)
constexpr int NBP = NB + 1;   // row pitch in float2: 26 words, conflict-free for 64-bit accesses down a column

//
// Variable-length batch (VARLEN): utterance b's output is its first Lb = clamp(lengths[b], 1, L) samples (all L when
// lengths is null), computed from its first Tb = min(T, 1 + Lb / hop) frames only; frames at or past Tb are staged
// as zeros, so a valid frame's pair partner is what a stand-alone call at (Lb, Tb) gives it.  CTAs keep their
// sample ranges, so samples below Lb are bit-identical to that call; samples in [Lb, L) are stored as 0, and a CTA
// wholly past Lb stores its zeros without staging or transforming anything.
template <bool VARLEN>
__global__ void istft_masked_kernel(const float2* __restrict__ spec, const float* __restrict__ masks, int S, int nfft,
                                    int log2n, int hop, int T, int F, int L, int CH, float* __restrict__ out,
                                    const int* __restrict__ lengths) {
  extern __shared__ __align__(16) uint8_t sm_raw[];
  double* win = reinterpret_cast<double*>(sm_raw);          // [nfft]
  double* acc = win + nfft;                                 // [CH]
  float2* tile = reinterpret_cast<float2*>(acc + CH);       // [F][NBP]
  float* re = reinterpret_cast<float*>(tile + static_cast<size_t>(F) * NBP);   // [nfft]
  float* im = re + nfft;                                    // [nfft]
  float* twr = im + nfft;                                   // [nfft/2]
  float* twi = twr + nfft / 2;                              // [nfft/2]
  const int b = blockIdx.z, s = blockIdx.y;
  const int n0 = blockIdx.x * CH;
  const int Lb = VARLEN ? clamp_len(lengths, b, L) : L;
  const int Tb = VARLEN ? min(T, 1 + Lb / hop) : T;
  const int n1 = min(n0 + CH, Lb);
  const int tid = threadIdx.x;
  if (VARLEN && n0 >= Lb) {                                 // CTA-uniform: nothing of this utterance here
    float* y = out + (static_cast<size_t>(b) * S + s) * L;
    for (int n = n0 + tid; n < min(n0 + CH, L); n += blockDim.x) y[n] = 0.f;
    return;
  }
  {
    float sv, cv;
    sincospif(2.0f * static_cast<float>(tid) / static_cast<float>(nfft), &sv, &cv);   // inverse: conj twiddles
    twr[tid] = cv; twi[tid] = sv;
    win[tid] = hann(tid, nfft);
    win[tid + nfft / 2] = hann(tid + nfft / 2, nfft);
  }
  for (int i = tid; i < CH; i += blockDim.x) acc[i] = 0.0;
  // frames overlapping [n0, n1): i*hop <= n1-1 and i*hop + nfft - 1 >= n0
  const int first = n0 - nfft + 1;
  const int i_lo = first > 0 ? (first + hop - 1) / hop : 0;
  const int i_hi = min(Tb - 1, (n1 - 1) / hop);
  const float2* X = spec + static_cast<size_t>(b) * F * T;
  const float* Mk = masks ? masks + (static_cast<size_t>(b) * S + s) * F * T : nullptr;
  const float inv_n = 1.0f / static_cast<float>(nfft);
  for (int ib = i_lo; ib <= i_hi; ib += NB) {
    const int nb = min(NB, i_hi - ib + 1);
    __syncthreads();
    for (int e = tid; e < F * NB; e += blockDim.x) {
      const int f = e / NB, j = e - f * NB;
      float2 v = make_float2(0.f, 0.f);
      if (j < nb) {
        const size_t o = static_cast<size_t>(f) * T + ib + j;
        v = X[o];
        if (Mk) { const float m = Mk[o]; v.x *= m; v.y *= m; }
        if (f == 0 || f == nfft / 2) v.y = 0.f;            // irfft ignores the imaginary part of DC and Nyquist
      }
      tile[f * NBP + j] = v;
    }
    for (int j = 0; j < nb; j += 2) {
      const int ia = ib + j;
      const bool has_b = j + 1 < nb;
      __syncthreads();
      // Z[k] = A[k] + i B[k] with A, B the Hermitian extensions of the two half spectra (frame b is zero when
      // absent); bit-reversed placement for the in-place transform.
      for (int k = tid; k < nfft; k += blockDim.x) {
        const int f = k <= nfft / 2 ? k : nfft - k;
        const float sgn = k <= nfft / 2 ? 1.f : -1.f;
        const float2 a = tile[f * NBP + j];
        const float2 bb = tile[f * NBP + j + 1];           // column NB is never written past nb: j + 1 <= NB - 1
        const int r = static_cast<int>(__brev(static_cast<unsigned>(k)) >> (32 - log2n));
        re[r] = a.x - sgn * bb.y;
        im[r] = sgn * a.y + bb.x;
      }
      fft_stages(re, im, twr, twi, log2n, tid);
      // overlap-add frame a, then frame b (a barrier between: the two frames hit the same samples hop apart)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k = tid + h * (nfft / 2);
        const int nn = ia * hop + k - n0;
        if (nn >= 0 && nn < n1 - n0) acc[nn] += win[k] * static_cast<double>(re[k] * inv_n);
      }
      if (has_b) {
        __syncthreads();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int k = tid + h * (nfft / 2);
          const int nn = (ia + 1) * hop + k - n0;
          if (nn >= 0 && nn < n1 - n0) acc[nn] += win[k] * static_cast<double>(im[k] * inv_n);
        }
      }
    }
  }
  __syncthreads();
  float* y = out + (static_cast<size_t>(b) * S + s) * L;
  for (int i = tid; i < n1 - n0; i += blockDim.x) {
    const int n = n0 + i;
    const int fl = n - nfft + 1;
    double wss = 0.0;
    for (int fr = fl > 0 ? (fl + hop - 1) / hop : 0; fr <= min(Tb - 1, n / hop); ++fr) {
      const double w = win[n - fr * hop];
      wss += w * w;
    }
    y[n] = wss > 1e-11 ? static_cast<float>(acc[i] / wss) : 0.f;
  }
  if (VARLEN)
    for (int n = n1 + tid; n < min(n0 + CH, L); n += blockDim.x) y[n] = 0.f;
}

// ---- n_fft = 512 (the reference's default geometry): register radix-8 transforms, fft512.cuh ----------------------
//
// 256 threads = 4 groups of 64; each group transforms one frame pair, so a CTA covers 8 frames in one pass.  The fp64
// Hann window and the twiddle tables live in device globals filled once per device (fft512_init_tables, called by
// avsep_create): evaluating 512 fp64 cosines per CTA was a fifth of the instructions of these kernels.
__device__ double g_hann512[512];
__device__ float2 g_tw512[FFT512_TW];

__global__ void fft512_tables_kernel() {
  const int tid = threadIdx.x;
  for (int k = tid; k < 512; k += blockDim.x) g_hann512[k] = hann(k, 512);
  fft512_fill_twiddles(g_tw512, tid, blockDim.x);
}

__device__ __forceinline__ void fft512_load_twiddles(float2* tw, int tid) {
  for (int m = tid; m < FFT512_TW; m += 256) tw[m] = g_tw512[m];
}

// grid (ceil(T/8), number of signals).  Output selection: S1 == 0 -> spec / mag indexed by signal; S1 > 0 (the
// synthesis layout, signals (B, S1) with the mixture first) -> magnitudes only, mag = mixed_spec (B, F, T) and
// mag2 = clean_specs (B, S1-1, F, T) or null.  VARLEN (S1 == 0 only): the variable-length rule of
// stft_complex_kernel; pairs are (t0 + 2g, t0 + 2g + 1), again fixed by absolute frame index.
template <bool VARLEN>
__global__ void __launch_bounds__(256) stft512_kernel(const float* __restrict__ waves, int n, int hop, int T,
                                                      float2* __restrict__ spec, float* __restrict__ mag,
                                                      float* __restrict__ mag2, int S1,
                                                      const int* __restrict__ lengths, int* __restrict__ frame_lengths) {
  constexpr int NF = 512, F = 257;
  extern __shared__ __align__(16) uint8_t sm_raw[];
  float2* tw = reinterpret_cast<float2*>(sm_raw);                  // [FFT512_TW]
  float2* stage = tw + FFT512_TW;                                  // [F][9] (pitch 9: conflict-free column writes)
  float* xch = reinterpret_cast<float*>(stage + F * 9);            // [4 groups][2 planes][FFT512_XCH]
  const int sig = blockIdx.y;
  const int t0 = blockIdx.x * 8;
  const int tid = threadIdx.x, g = tid >> 6, t = tid & 63;
  const float* x = waves + static_cast<size_t>(sig) * n;
  const int nb = VARLEN ? clamp_len(lengths, sig, n) : n;          // this utterance's samples and frames
  const int Tb = VARLEN ? 1 + nb / hop : T;
  if (VARLEN && frame_lengths && blockIdx.x == 0 && tid == 0) frame_lengths[sig] = Tb;
  if (!VARLEN || t0 < Tb) {             // CTA-uniform: a CTA wholly past Tb only stores zeros
    fft512_load_twiddles(tw, tid);
    __syncthreads();
    const int ng = min(8, Tb - t0);
    const int ta = t0 + 2 * g;
    const bool has_a = 2 * g < ng, has_b = 2 * g + 1 < ng;
    float* xr = xch + g * 2 * FFT512_XCH;
    float* xi = xr + FFT512_XCH;
    float2 v[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int k = t + 64 * q;
      const int sa = ta * hop + k, sb = sa + hop;
      const float va = (has_a && sa < nb) ? x[sa] : 0.f;
      const float vb = (has_b && sb < nb) ? x[sb] : 0.f;
      const double w = g_hann512[k];
      v[q] = make_float2(static_cast<float>(static_cast<double>(va) * w),     // float32 `frame *= window`
                         static_cast<float>(static_cast<double>(vb) * w));
    }
    fft512_regs<-1>(v, t, xr, xi, tw);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) {          // natural order (padded): k = hi + 8 lo + 64 i
      const int k = fft512_nat(fft512_out_index(t, i));
      xr[k] = v[i].x; xi[k] = v[i].y;
    }
    __syncthreads();
    for (int f = t; f < F; f += 64) {
      const int kf = fft512_nat(f), kn = fft512_nat((NF - f) & (NF - 1));
      const float zr = xr[kf], zi = xi[kf], yr = xr[kn], yi = xi[kn];
      if (has_a) stage[f * 9 + 2 * g] = make_float2(0.5f * (zr + yr), 0.5f * (zi - yi));       // A = (Z + conj Z~)/2
      if (has_b) stage[f * 9 + 2 * g + 1] = make_float2(0.5f * (zi + yi), 0.5f * (yr - zr));   // B = (Z - conj Z~)/2i
    }
    __syncthreads();
  }
  const int ng = min(8, Tb - t0);
  float* m_out = mag;
  size_t base = static_cast<size_t>(sig) * F * T;
  if (S1 > 0) {
    const int b = sig / S1, j = sig - b * S1;
    m_out = j == 0 ? mag : mag2;
    base = j == 0 ? static_cast<size_t>(b) * F * T : (static_cast<size_t>(b) * (S1 - 1) + (j - 1)) * F * T;
  }
  for (int e = tid; e < F * 8; e += 256) {
    const int f = e >> 3, gg = e & 7;
    if (gg >= (VARLEN ? T - t0 : ng)) continue;
    const size_t o = base + static_cast<size_t>(f) * T + t0 + gg;
    const float2 z = (!VARLEN || gg < ng) ? stage[f * 9 + gg] : make_float2(0.f, 0.f);
    if (spec) spec[o] = z;
    if (m_out) m_out[o] = 0.5f * hypotf(2.0f * z.x, 2.0f * z.y);
  }
}

// grid (ceil(L/CH), S, B), CH = (9 - R) * hop with R = ceil(512 / hop) <= 8: exactly the (at most) 8 frames
// i_first .. i_first + 7 overlap the CTA's samples.  Their masked half spectra are staged once (row-contiguous
// loads), each group inverts one pair, the 8 time frames replace the staged tile, and every output sample gathers
// its frames in ascending order (deterministic, no atomics).  VARLEN: the variable-length rule of istft_masked_kernel.
template <bool VARLEN>
__global__ void __launch_bounds__(256) istft512_kernel(const float2* __restrict__ spec, const float* __restrict__ masks,
                                                       int S, int hop, int T, int L, int CH, int R,
                                                       float* __restrict__ out, const int* __restrict__ lengths) {
  constexpr int NF = 512, F = 257, NBP8 = 9;   // pitch 18 words: conflict-free 64-bit accesses down a column
  extern __shared__ __align__(16) uint8_t sm_raw[];
  float2* tw = reinterpret_cast<float2*>(sm_raw);                  // [FFT512_TW]
  float* xch = reinterpret_cast<float*>(tw + FFT512_TW);           // [4][2][FFT512_XCH]
  float2* tile = reinterpret_cast<float2*>(xch + 8 * FFT512_XCH);  // [F][NBP8]; later float frames[8][FFT512_XCH]
  float* frames = reinterpret_cast<float*>(tile);
  const int b = blockIdx.z, s = blockIdx.y;
  const int n0 = blockIdx.x * CH;
  const int Lb = VARLEN ? clamp_len(lengths, b, L) : L;
  const int Tb = VARLEN ? min(T, 1 + Lb / hop) : T;
  const int n1 = min(n0 + CH, Lb);
  const int tid = threadIdx.x, g = tid >> 6, t = tid & 63;
  if (VARLEN && n0 >= Lb) {                                        // CTA-uniform: nothing of this utterance here
    float* y = out + (static_cast<size_t>(b) * S + s) * L;
    for (int n = n0 + tid; n < min(n0 + CH, L); n += 256) y[n] = 0.f;
    return;
  }
  const int i_first = n0 / hop - (R - 1);                          // may be negative: those frames do not exist
  fft512_load_twiddles(tw, tid);
  const float2* X = spec + static_cast<size_t>(b) * F * T;
  const float* Mk = masks ? masks + (static_cast<size_t>(b) * S + s) * F * T : nullptr;
  {
    // thread -> (frame column j, rows f0 + 32 it): 8 consecutive threads read the 64 contiguous bytes of one bin's
    // frames; loads are issued three rows ahead of their use so that six are in flight per thread
    const int j = tid & 7, f0 = tid >> 3;
    const int fr = i_first + j;
    const bool fr_ok = fr >= 0 && fr < Tb;
    const float2* Xp = X + (fr_ok ? fr : 0);
    const float* Mp = Mk ? Mk + (fr_ok ? fr : 0) : nullptr;
#pragma unroll
    for (int it0 = 0; it0 < 9; it0 += 3) {
      float2 z[3];
      float m[3];
#pragma unroll
      for (int u = 0; u < 3; ++u) {
        const int f = f0 + 32 * (it0 + u);
        const bool ok = fr_ok && f < F;
        z[u] = ok ? __ldg(Xp + static_cast<size_t>(f) * T) : make_float2(0.f, 0.f);
        m[u] = (ok && Mp) ? __ldg(Mp + static_cast<size_t>(f) * T) : 1.f;
      }
#pragma unroll
      for (int u = 0; u < 3; ++u) {
        const int f = f0 + 32 * (it0 + u);
        float2 zz = make_float2(z[u].x * m[u], z[u].y * m[u]);
        if (f == 0 || f == NF / 2) zz.y = 0.f;                     // irfft ignores the imaginary part of DC / Nyquist
        if (f < F) tile[f * NBP8 + j] = zz;
      }
    }
  }
  __syncthreads();
  float* xr = xch + g * 2 * FFT512_XCH;
  float* xi = xr + FFT512_XCH;
  float2 v[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {          // Z[k] = A[k] + i B[k], Hermitian extensions of the pair (2g, 2g+1)
    const int k = t + 64 * q;
    const int f = k <= NF / 2 ? k : NF - k;
    const float sgn = k <= NF / 2 ? 1.f : -1.f;
    const float2 a = tile[f * NBP8 + 2 * g];
    const float2 bb = tile[f * NBP8 + 2 * g + 1];
    v[q] = make_float2(a.x - sgn * bb.y, sgn * a.y + bb.x);
  }
  fft512_regs<1>(v, t, xr, xi, tw);      // its barriers also order the tile reads above before the overwrite below
  const float inv_n = 1.0f / static_cast<float>(NF);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int k = fft512_nat(fft512_out_index(t, i));
    frames[(2 * g) * FFT512_XCH + k] = v[i].x * inv_n;
    frames[(2 * g + 1) * FFT512_XCH + k] = v[i].y * inv_n;
  }
  __syncthreads();
  float* y = out + (static_cast<size_t>(b) * S + s) * L;
  for (int i = tid; i < n1 - n0; i += 256) {
    const int n = n0 + i;
    double acc = 0.0, wss = 0.0;
    // frames covering n: fr*hop <= n < fr*hop + 512, ascending
    const int fr_hi = min(n / hop, Tb - 1);
    const int below = n - NF + 1;
    for (int fr = max(max(below > 0 ? (below + hop - 1) / hop : 0, i_first), 0); fr <= fr_hi; ++fr) {
      const int k = n - fr * hop;
      const double w = g_hann512[k];
      acc += w * static_cast<double>(frames[(fr - i_first) * FFT512_XCH + fft512_nat(k)]);
      wss += w * w;
    }
    y[n] = wss > 1e-11 ? static_cast<float>(acc / wss) : 0.f;
  }
  if (VARLEN)
    for (int n = n1 + tid; n < min(n0 + CH, L); n += 256) y[n] = 0.f;
}

constexpr size_t kStft512Smem = FFT512_TW * sizeof(float2) + 257 * 9 * sizeof(float2) + 8 * FFT512_XCH * sizeof(float);
constexpr size_t kIstft512Smem = FFT512_TW * sizeof(float2) + 8 * FFT512_XCH * sizeof(float) + 257 * 9 * sizeof(float2);
static_assert(257 * 9 * sizeof(float2) >= 8 * FFT512_XCH * sizeof(float), "the time frames must fit in the staged tile");
static_assert(kStft512Smem <= 48 * 1024 && kIstft512Smem <= 48 * 1024, "no opt-in shared memory needed");

bool fft_geometry_ok(int nfft, int hop, int* log2n) {
  if (nfft < 8 || nfft > 2048 || (nfft & (nfft - 1)) || hop < 1 || hop > nfft) return false;
  *log2n = 0;
  while ((1 << *log2n) < nfft) ++*log2n;
  return true;
}

}  // namespace

const char* fft512_init_tables() {
  fft512_tables_kernel<<<1, 256>>>();
  if (cudaGetLastError() != cudaSuccess) return "fft512: table kernel launch failed";
  return cudaDeviceSynchronize() == cudaSuccess ? nullptr : "fft512: table kernel failed";
}

const char* launch_stft_complex(cudaStream_t s, const float* waves, const int* lengths, int B, int L, int nfft, int hop,
                                float* spec, float* mag, int* frame_lengths) {
  int log2n;
  if (B <= 0 || L <= 0) return "stft: empty problem";
  if (!fft_geometry_ok(nfft, hop, &log2n)) return "stft: n_fft must be a power of two in [8, 2048], 1 <= hop <= n_fft";
  const int T = 1 + L / hop, F = nfft / 2 + 1;
  const bool varlen = lengths || frame_lengths;
  if (nfft == 512 && B <= 65535) {
    auto kern = varlen ? stft512_kernel<true> : stft512_kernel<false>;
    kern<<<dim3((T + 7) / 8, B), 256, kStft512Smem, s>>>(waves, L, hop, T, reinterpret_cast<float2*>(spec), mag,
                                                         nullptr, 0, lengths, frame_lengths);
    return cudaGetLastError() == cudaSuccess ? nullptr : "stft: launch failed";
  }
  const size_t smem = static_cast<size_t>(nfft) * sizeof(double) + 3 * static_cast<size_t>(nfft) * sizeof(float) +
                      static_cast<size_t>(F) * TGA * sizeof(float2);
  auto kern = varlen ? stft_complex_kernel<true> : stft_complex_kernel<false>;
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
    return "stft: cannot raise the shared-memory limit";
  kern<<<dim3((T + TGA - 1) / TGA, B), nfft / 2, smem, s>>>(waves, L, nfft, log2n, hop, T, F,
                                                           reinterpret_cast<float2*>(spec), mag, lengths, frame_lengths);
  return cudaGetLastError() == cudaSuccess ? nullptr : "stft: launch failed";
}

// Magnitude-only analysis of the synthesis layout (signals (B, S+1, n), mixture first) for n_fft = 512: used by
// launch_synth instead of its radix-2 kernel.
const char* launch_stft512_synth(cudaStream_t s, const float* waves, int B, int S, int n, int hop, float* mixed_spec,
                                 float* clean_specs) {
  const int T = 1 + n / hop;
  if (static_cast<long long>(B) * (S + 1) > 65535) return "synth: batch * (speakers + 1) above 65535";
  stft512_kernel<false><<<dim3((T + 7) / 8, B * (S + 1)), 256, kStft512Smem, s>>>(waves, n, hop, T, nullptr, mixed_spec,
                                                                                  clean_specs, S + 1, nullptr, nullptr);
  return cudaGetLastError() == cudaSuccess ? nullptr : "synth: stft launch failed";
}

const char* launch_istft_masked(cudaStream_t s, const float* spec, const float* masks, const int* lengths, int B, int S,
                                int T, int nfft, int hop, int L, float* waves) {
  int log2n;
  if (B <= 0 || S <= 0 || T <= 0 || L <= 0) return "istft: empty problem";
  if (!fft_geometry_ok(nfft, hop, &log2n)) return "istft: n_fft must be a power of two in [8, 2048], 1 <= hop <= n_fft";
  if (S > 65535 || B > 65535) return "istft: batch or speaker count above 65535";
  if (masks == nullptr && S != 1) return "istft: without masks there is one output per utterance (S = 1)";
  if (static_cast<long long>(T - 1) * hop + nfft < L) return "istft: the frames do not reach the requested length";
  const int F = nfft / 2 + 1;
  if (nfft == 512 && hop >= 64) {
    const int R = (512 + hop - 1) / hop, CH = (9 - R) * hop;
    auto kern = lengths ? istft512_kernel<true> : istft512_kernel<false>;
    kern<<<dim3((L + CH - 1) / CH, S, B), 256, kIstft512Smem, s>>>(reinterpret_cast<const float2*>(spec), masks, S, hop,
                                                                   T, L, CH, R, waves, lengths);
    return cudaGetLastError() == cudaSuccess ? nullptr : "istft: launch failed";
  }
  int tg = 4096 / hop;
  tg = tg < 1 ? 1 : (tg > 8 ? 8 : tg);
  const int CH = tg * hop;
  const size_t smem = (static_cast<size_t>(nfft) + CH) * sizeof(double) + static_cast<size_t>(F) * NBP * sizeof(float2) +
                      3 * static_cast<size_t>(nfft) * sizeof(float);
  if (smem > 227 * 1024) return "istft: geometry needs more than 227 KB of shared memory";
  auto kern = lengths ? istft_masked_kernel<true> : istft_masked_kernel<false>;
  // per call, not cached: the attribute is per device and a process may hold engines on several
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
    return "istft: cannot raise the shared-memory limit";
  kern<<<dim3((L + CH - 1) / CH, S, B), nfft / 2, smem, s>>>(reinterpret_cast<const float2*>(spec), masks, S, nfft,
                                                             log2n, hop, T, F, L, CH, waves, lengths);
  return cudaGetLastError() == cudaSuccess ? nullptr : "istft: launch failed";
}

}  // namespace avsep
