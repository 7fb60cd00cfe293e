// Log-mel front-end (SURVEY.md 8(f) rank 2): FilterbankFeatures.forward in eval mode
// (nemo/collections/asr/parts/preprocessing/features.py:358-453) for the configuration of the Conformer recipes --
// pre-emphasis, centred STFT with reflect padding (n_fft = 512), |.|^2, mel projection, log(x + guard), per-feature
// mean / std normalisation over the valid frames, zero padding of the rest.
//
//   logmel_frames_kernel     one warp per frame: the 512 windowed, pre-emphasised real samples are packed as 256 complex
//                            values (bit-reversed) in a private shared-memory buffer, eight radix-2 stages (4
//                            butterflies per lane, twiddles from a 256-entry table in shared memory), one untangling
//                            pass to the 257 bins of the real transform and their power, then every lane owns mel bins
//                            lane, lane + 32, lane + 64 and walks only the FFT bins its triangular filter covers
//                            (spans found once on the host).  A CTA's 16 frames are staged as a (mel, frame) tile and
//                            written as 64-byte row segments.
//   logmel_normalize_kernel  one warp per (utterance, mel bin) row: mean, unbiased std + 1e-5 over the valid frames
//                            (two passes over a row that the first kernel just left in L2), normalised in place,
//                            zeros from seq_len on; also writes seq_len = floor(len / hop) + 1 computed in float32
//                            like features.py:347-353.  With normalisation off (normalize: "None", the buffered
//                            long-audio front end) the same kernel only writes seq_len and zeroes the tail.
// Both are bandwidth-trivial next to the encoder (640 s of audio: 41 MB in, 20 MB out); no tensor cores on purpose.
#include <math.h>
#include <stdio.h>

#include "common.cuh"

namespace cfb {

namespace {

constexpr int kNfft = 512;
constexpr int kBins = kNfft / 2 + 1;
constexpr int kFramesPerCta = 16;
constexpr int kWarps = 8;
constexpr int kMaxMels = 96;  // three mel bins per lane

__device__ __forceinline__ int bitrev8(int v) { return static_cast<int>(__brev(static_cast<unsigned>(v)) >> 24); }

__global__ void __launch_bounds__(32 * kWarps)
logmel_frames_kernel(const float* __restrict__ audio, int L, const float* __restrict__ window, int win_length, int hop,
                     const float* __restrict__ fb, const int* __restrict__ fb_span, int n_mels, float preemph,
                     float log_guard, float* __restrict__ feat, int T, int T_out) {
  // per warp: z[256] (the packed half-size FFT) followed by the 257 power values (the second half of the buffer)
  __shared__ float2 buf[kWarps][kNfft];
  __shared__ float2 tw[kNfft / 2];  // W_512^k, k < 256
  __shared__ float tile[kMaxMels][kFramesPerCta + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * kFramesPerCta;
  for (int k = threadIdx.x; k < kNfft / 2; k += blockDim.x) {
    float sn, cs;
    sincospif(-2.0f * static_cast<float>(k) / kNfft, &sn, &cs);
    tw[k] = make_float2(cs, sn);
  }
  // this lane's mel bins (lane, lane + 32, lane + 64): first FFT bin and number of bins of each triangular filter
  int m_start[3], m_len[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const int m = lane + 32 * j;
    m_start[j] = m < n_mels ? __ldg(fb_span + 2 * m) : 0;
    m_len[j] = m < n_mels ? __ldg(fb_span + 2 * m + 1) : 0;
  }
  pdl_launch_dependents();
  pdl_wait();
  __syncthreads();
  const float* x = audio + static_cast<long long>(b) * L;
  const int w_off = (kNfft - win_length) / 2;  // torch.stft centres a short window inside n_fft
  float2* z = buf[warp];
  float* pwr = reinterpret_cast<float*>(buf[warp] + kNfft / 2);
  // windowed sample n of frame t of the pre-emphasised, reflect-padded signal (features.py:371-376; center = True pads
  // n_fft / 2 samples on both sides of the WHOLE row)
  auto sample = [&](int t, int n) -> float {
    const int wn = n - w_off;
    if (wn < 0 || wn >= win_length) return 0.f;
    int s = t * hop - kNfft / 2 + n;
    if (s < 0) s = -s;
    if (s >= L) s = 2 * (L - 1) - s;
    s = min(max(s, 0), L - 1);
    const float cur = __ldg(x + s);
    const float y = s > 0 ? cur - preemph * __ldg(x + s - 1) : cur;
    return y * __ldg(window + wn);
  };
  for (int f = warp; f < kFramesPerCta; f += kWarps) {
    const int t = t0 + f;
    if (t >= T) break;  // warp-uniform
    // ---- real 512-point DFT through a 256-point complex FFT of z[n] = x[2n] + i x[2n+1] (bit-reversed store)
    for (int n = lane; n < kNfft / 2; n += 32) z[bitrev8(n)] = make_float2(sample(t, 2 * n), sample(t, 2 * n + 1));
    __syncwarp();
#pragma unroll 1
    for (int half = 1; half < kNfft / 2; half <<= 1) {
      const int tstep = (kNfft / 2) / half;  // W_256^j = W_512^(2j): index j * 256 / half into the 512-table
#pragma unroll
      for (int q = lane; q < kNfft / 4; q += 32) {
        const int j = q & (half - 1);
        const int i = ((q - j) << 1) + j;
        const float2 w = tw[j * tstep];
        const float2 a = z[i], c = z[i + half];
        const float2 wc = make_float2(w.x * c.x - w.y * c.y, w.x * c.y + w.y * c.x);
        z[i] = make_float2(a.x + wc.x, a.y + wc.y);
        z[i + half] = make_float2(a.x - wc.x, a.y - wc.y);
      }
      __syncwarp();
    }
    // ---- untangle: X[k] = E[k] + W_512^k O[k], E = (Z[k] + conj Z[256-k]) / 2, O = (Z[k] - conj Z[256-k]) / (2i); the
    // reference takes sqrt(re^2 + im^2) and squares it again (features.py:385, 393-394)
    for (int k = lane; k < kNfft / 2; k += 32) {
      const float2 zk = z[k], zn = z[(kNfft / 2 - k) & (kNfft / 2 - 1)];
      const float2 e = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
      const float2 o = make_float2(0.5f * (zk.y + zn.y), -0.5f * (zk.x - zn.x));
      const float2 w = tw[k];
      const float re = e.x + (w.x * o.x - w.y * o.y), im = e.y + (w.x * o.y + w.y * o.x);
      const float mag = sqrtf(re * re + im * im);
      pwr[k] = mag * mag;
      if (k == 0) {
        const float nyq = fabsf(zk.x - zk.y);  // X[256] = E[0] - O[0], purely real
        pwr[kNfft / 2] = nyq * nyq;
      }
    }
    __syncwarp();
    // ---- mel projection over each filter's own bins + log (features.py:397-402)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int m = lane + 32 * j;
      if (m < n_mels) {
        const float* row = fb + static_cast<long long>(m) * kBins + m_start[j];
        const float* pp = pwr + m_start[j];
        float acc = 0.f;
        for (int k = 0; k < m_len[j]; ++k) acc = fmaf(__ldg(row + k), pp[k], acc);
        tile[m][f] = logf(acc + log_guard);
      }
    }
    __syncwarp();
  }
  __syncthreads();
  const int nf = min(kFramesPerCta, T - t0);
  for (int i = threadIdx.x; i < n_mels * kFramesPerCta; i += blockDim.x) {
    const int m = i / kFramesPerCta, f = i % kFramesPerCta;
    if (f < nf) feat[(static_cast<long long>(b) * n_mels + m) * T_out + t0 + f] = tile[m][f];
  }
}

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(256)
logmel_normalize_kernel(float* __restrict__ feat, const long long* __restrict__ lengths, int n_rows, int n_mels, int T,
                        int T_out, int hop, bool normalize, float std_eps, long long* __restrict__ seq_len_out,
                        int* __restrict__ flag) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();
  if (row >= n_rows) return;
  const int b = row / n_mels;
  // features.py:347-353 with center = True: floor((len + 2 (n_fft/2) - n_fft) / hop) + 1 in float32
  const float lf = static_cast<float>(lengths[b]);
  long long n_ll = static_cast<long long>(floorf(__fdiv_rn(__fadd_rn(__fadd_rn(lf, static_cast<float>(kNfft)), -static_cast<float>(kNfft)),
                                                           static_cast<float>(hop)))) + 1;
  if (row % n_mels == 0 && lane == 0) {
    seq_len_out[b] = n_ll;
    if (normalize && n_ll == 1) atomicExch(flag, 1);  // the reference raises: std of one frame is NaN (features.py:58-62)
  }
  const int n = static_cast<int>(n_ll < 0 ? 0 : (n_ll > T ? T : n_ll));
  float* r = feat + static_cast<long long>(row) * T_out;
  if (!normalize) {  // normalize_batch returns x unchanged; frames from seq_len on are still set to pad_value (0)
    for (int t = n + lane; t < T_out; t += 32) r[t] = 0.f;
    return;
  }
  float s = 0.f;
  for (int t = lane; t < n; t += 32) s += r[t];
  const float mean = warp_sum_f(s) / static_cast<float>(n);
  float q = 0.f;
  for (int t = lane; t < n; t += 32) {
    const float d = r[t] - mean;
    q = fmaf(d, d, q);
  }
  const float stdv = sqrtf(warp_sum_f(q) / static_cast<float>(n - 1)) + std_eps;
  for (int t = lane; t < T_out; t += 32) r[t] = t < n ? (r[t] - mean) / stdv : 0.f;
}

}  // namespace

int launch_logmel(const LogMelDesc& d, cudaStream_t st, std::string* err) {
  if (d.B <= 0 || d.L <= 0) return 0;
  if (d.n_fft != kNfft || d.win_length < 1 || d.win_length > kNfft || d.hop < 1 || d.n_mels < 1 || d.n_mels > kMaxMels) {
    if (err) *err = "logmel: n_fft must be 512, win_length <= 512, hop >= 1, n_mels <= 96";
    return -1;
  }
  if (d.L <= kNfft / 2) {
    if (err) *err = "logmel: reflect padding needs more than n_fft / 2 samples per row";
    return -1;
  }
  const int T = 1 + d.L / d.hop;  // torch.stft, center = True
  if (d.T_out < T) {
    if (err) *err = "logmel: T_out is smaller than 1 + L / hop";
    return -1;
  }
  if (d.normalize) {
    cudaError_t e = cudaMemsetAsync(d.flag, 0, sizeof(int), st);
    if (e != cudaSuccess) return static_cast<int>(e);
  }
  launch_pdl(logmel_frames_kernel, dim3((T + kFramesPerCta - 1) / kFramesPerCta, d.B), dim3(32 * kWarps), 0, st, d.audio, d.L,
             d.window, d.win_length, d.hop, d.fb, d.fb_span, d.n_mels, d.preemph, d.log_guard, d.features, T, d.T_out);
  const int rows = d.B * d.n_mels;
  launch_pdl(logmel_normalize_kernel, dim3((rows + 7) / 8), dim3(256), 0, st, d.features,
             reinterpret_cast<const long long*>(d.lengths), rows, d.n_mels, T, d.T_out, d.hop, d.normalize, d.std_eps,
             reinterpret_cast<long long*>(d.seq_len), d.flag);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace cfb
