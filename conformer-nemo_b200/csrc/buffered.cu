// Buffered long-audio inference (nemo/collections/asr/parts/utils/streaming_utils.py:455-684): the windows that
// FeatureFrameBufferer builds from the raw log-mel features of a file, for many files in one launch.
//
//   feature_buffers_kernel  one warp per (window, mel row), eight rows per CTA.  Column j of window k of a file with n
//                           valid frames is stream frame s = (k + 1) * fl - W + j: the silence level Z = -16.635 while
//                           s < 0 (the buffer starts filled with it), the feature X[:, s] while s < n, zero after (the
//                           last chunk is zero-filled past n).  The row is normalised on its own statistics: mean and
//                           population std (np.mean / np.std, ddof 0) over all W columns, (x - mean) / (std + 1e-5).
// The statistics are reduced lane-strided and then by a fixed butterfly, so a window's output does not depend on the
// other files of the call.  Memory-bound: the windows it writes are W / fl times the features it reads.
#include "common.cuh"

namespace cfb {

namespace {

constexpr float kSilence = -16.635f;  // ZERO_LEVEL_SPEC_DB_VAL: the log-mel value of a zero signal (preprocessor.log)
constexpr float kStdEps = 1e-5f;      // CONSTANT of normalize_frame_buffers
constexpr int kRows = 8;              // warps (mel rows) per CTA

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// NPL > 0: each lane keeps its columns j = lane + 32 i (i < NPL, W <= 32 NPL) in registers, so all loads of a row are in
// flight at once; NPL == 0: any W, three passes over the row.  Both sum in the same order (lane-strided, then the
// butterfly) and give the same bits.
template <int NPL>
__global__ void __launch_bounds__(32 * kRows)
feature_buffers_kernel(const float* __restrict__ feat, int n_files, int F, int T, const long long* __restrict__ seq_len,
                       const int* __restrict__ first_window, int fl, int W, float* __restrict__ out) {
  const int w = blockIdx.x;
  const int m = blockIdx.y * kRows + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (m >= F) return;
  // the file of window w: the last f with first_window[f] <= w
  int lo = 0, hi = n_files - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(first_window + mid) <= w) lo = mid;
    else hi = mid - 1;
  }
  const long long k = w - __ldg(first_window + lo);
  const long long n = min(__ldg(seq_len + lo), static_cast<long long>(T));
  const float* x = feat + (static_cast<long long>(lo) * F + m) * T;
  const long long s0 = (k + 1) * fl - W;
  auto column = [&](int j) -> float {
    const long long s = s0 + j;
    return s < 0 ? kSilence : (s < n ? __ldg(x + s) : 0.f);
  };
  float* o = out + (static_cast<long long>(w) * F + m) * W;
  float sum = 0.f, q = 0.f;
  if constexpr (NPL > 0) {
    float v[NPL];
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int j = lane + 32 * i;
      v[i] = j < W ? column(j) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < NPL; ++i) sum += v[i];  // + 0 for the columns past W: the same bits as the loop below
    const float mean = warp_sum(sum) / static_cast<float>(W);
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const float d = v[i] - mean;
      if (lane + 32 * i < W) q = fmaf(d, d, q);
    }
    const float denom = sqrtf(warp_sum(q) / static_cast<float>(W)) + kStdEps;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int j = lane + 32 * i;
      if (j < W) o[j] = (v[i] - mean) / denom;
    }
  } else {
    for (int j = lane; j < W; j += 32) sum += column(j);
    const float mean = warp_sum(sum) / static_cast<float>(W);
    for (int j = lane; j < W; j += 32) {
      const float d = column(j) - mean;
      q = fmaf(d, d, q);
    }
    const float denom = sqrtf(warp_sum(q) / static_cast<float>(W)) + kStdEps;
    for (int j = lane; j < W; j += 32) o[j] = (column(j) - mean) / denom;
  }
}

}  // namespace

int launch_feature_buffers(const float* feat, int n_files, int F, int T, const long long* seq_len, const int* first_window,
                           int n_windows, int fl, int W, float* out, cudaStream_t st, std::string* err) {
  if (n_windows == 0) return 0;
  if (n_files < 1 || F < 1 || T < 1 || n_windows < 0 || fl < 1 || W < fl) {
    if (err) *err = "feature_buffers: needs n_files, F, T >= 1 and 1 <= frame_len <= buffer_len";
    return -1;
  }
  const dim3 grid(n_windows, (F + kRows - 1) / kRows);
  auto kern = W <= 128 ? feature_buffers_kernel<4> : W <= 256 ? feature_buffers_kernel<8>
            : W <= 512 ? feature_buffers_kernel<16> : W <= 1024 ? feature_buffers_kernel<32> : feature_buffers_kernel<0>;
  kern<<<grid, 32 * kRows, 0, st>>>(feat, n_files, F, T, seq_len, first_window, fl, W, out);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace cfb
