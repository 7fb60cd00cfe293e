// Packed (variable-length) batches: the device-side layout tables, the first conv's patch gather for the packed time
// axis and the LayerNorm that scatters the packed result back into the dense (B, T', d) tensor of the reference API
// (conformer_encoder.py:280).  See common.cuh (PackedTables) for the layout; engine.cu (forward_packed) for its use.
//
// Reference semantics reproduced exactly: the reference runs its strided convolutions over the PADDED batch
// (subsampling.py:172-175), so the last valid output frame of a short utterance sees relu(conv(0-extended input))
// of the frames behind it, while the longest utterance of the batch sees the convolution's zero padding.  The packed
// gather therefore computes first-conv rows t1 <= T1_b of every utterance from its zero-extended features (row T1_b is
// the only one behind the utterance a valid output reads) and writes zero rows for t1 >= T1 of the padded batch and for
// everything else in the gap -- which is also the zero row in FRONT of the next utterance.
#include "common.cuh"

namespace cfb {
namespace {

constexpr int kPlanThreads = 1024;

__device__ __forceinline__ int clip_len(const long long* lengths, int b, int T) {
  if (lengths == nullptr) return T;
  const long long v = lengths[b];
  return v < 0 ? 0 : (v > T ? T : static_cast<int>(v));
}

// One CTA.  The launch lays out the GROUP of utterances first, first + step, ... (B of them; the engine runs a batch as
// two interleaved groups on two streams).  Slot k of the group holds utterance first + k * step; tiles / row_out carry
// the utterance's index in the whole batch.
__global__ void __launch_bounds__(kPlanThreads) packed_plan_kernel(const long long* __restrict__ lengths, int B, int first,
                                                                   int step, int T, int T2, int n_rows, int n_tiles,
                                                                   PackedTables tb) {
  extern __shared__ int sh[];  // [B] slot rows -> exclusive prefix (row0), [B] query tiles -> exclusive prefix, [B] t2
  int* s_row0 = sh;
  int* s_tile0 = sh + B;
  int* s_t2 = sh + 2 * B;
  int* s_rows = sh + 3 * B;
  pdl_launch_dependents();
  pdl_wait();
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const int len = clip_len(lengths, first + b * step, T);
    const int t1 = (len + 1) >> 1;
    const int t2 = (t1 + 1) >> 1;
    const int rows = (t2 + kPackGap + kPackAlign - 1) / kPackAlign * kPackAlign;
    s_t2[b] = t2;
    s_rows[b] = rows;
  }
  __syncthreads();
  if (threadIdx.x == 0) {  // B is small (<= a few hundred): a serial scan costs less than it would to be clever
    int r = 0, q = 0;
    for (int b = 0; b < B; ++b) {
      s_row0[b] = r;
      s_tile0[b] = q;
      r += s_rows[b];
      q += (s_rows[b] + 127) / 128;
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    tb.seq_row0[b] = s_row0[b];
    tb.seq_rows[b] = s_rows[b];
    const int nq = (s_rows[b] + 127) / 128;
    for (int q = 0; q < nq; ++q)
      if (s_tile0[b] + q < n_tiles) tb.tiles[s_tile0[b] + q] = make_int4(first + b * step, q * 128, s_row0[b], s_rows[b]);
  }
  for (int r = threadIdx.x; r < n_rows; r += blockDim.x) {
    int lo = 0, hi = B - 1;  // last b with row0[b] <= r
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (s_row0[mid] <= r) lo = mid;
      else hi = mid - 1;
    }
    const int t = r - s_row0[lo];
    const bool valid = t < s_t2[lo];
    tb.row_t[r] = valid ? t : -1;
    tb.row_out[r] = valid ? (first + lo * step) * T2 + t : -1;
    if ((r & (kPackAlign - 1)) == 0) tb.blk_seq[r / kPackAlign] = lo;
  }
}

// ------------------------------------------------------------------------------------------------ conv 0 gather, packed
// Same row format as conv0_im2col_kernel (elementwise.cu): [x_hi (9) | x_lo (9) | 1 | 1 | 0 0 0 0] per output position,
// in the row order of the parity-split y1 of ONE virtual sequence of 2 * n_rows first-conv rows.
constexpr int kS1T = 16;  // t1 rows per block = kPackAlign token rows
static_assert((kMaxFeatIn + 2) * (2 * kS1T + 2) * sizeof(float) <= 48 * 1024, "feature patch must fit the default shared memory");
constexpr int kA0Cols = kConv0Cols;

template <typename TIn>
__global__ void __launch_bounds__(256) conv0_im2col_packed_kernel(const TIn* __restrict__ feats,
                                                                  const long long* __restrict__ lengths,
                                                                  bf16* __restrict__ a0, int first, int step, int F, int T,
                                                                  int T1, int F1, int Fh, int n_rows, PackedTables tb) {
  extern __shared__ float patch[];  // [F + 2][2*kS1T + 2]
  const int pw = 2 * kS1T + 2;
  pdl_launch_dependents();
  pdl_wait();
  const int blk = blockIdx.x;
  const int k = tb.blk_seq[blk];  // slot of the group
  const int b = first + k * step;  // utterance of the batch
  const int t1_0 = 2 * (blk * kPackAlign - tb.seq_row0[k]);  // first local first-conv row of this block
  const int len = clip_len(lengths, b, T);
  const int t1_live = min((len + 1) >> 1, T1 - 1);  // local rows 0 .. t1_live are computed, the rest are zero rows
  const TIn* xb = feats + static_cast<long long>(b) * F * T;
  const bool any_live = t1_0 <= t1_live;
  if (any_live) {
    for (int i = threadIdx.x; i < (F + 2) * (2 * kS1T + 1); i += 256) {
      const int fr = i / (2 * kS1T + 1), tc = i % (2 * kS1T + 1);
      const int f = fr - 1, t = 2 * t1_0 - 1 + tc;
      float v = 0.f;
      if (f >= 0 && f < F && t >= 0 && t < T) v = static_cast<float>(xb[static_cast<long long>(f) * T + t]);
      patch[fr * pw + tc] = v;
    }
  }
  __syncthreads();
  const int positions = kS1T * 2 * Fh;
  const long long Th = n_rows;  // plane extent of the virtual sequence
  for (int pos = threadIdx.x; pos < positions; pos += 256) {
    const int fh = pos % Fh;
    const int pf = (pos / Fh) & 1;
    const int tt = pos / (2 * Fh);
    const int f1 = 2 * fh + pf;
    const int t1 = t1_0 + tt;
    uint32_t w[kA0Cols / 2];
#pragma unroll
    for (int j = 0; j < kA0Cols / 2; ++j) w[j] = 0u;
    if (t1 <= t1_live && f1 < F1) {
      unsigned short hi[9], lo[9];
#pragma unroll
      for (int kh = 0; kh < 3; ++kh)
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          const float v = patch[(2 * f1 + kw) * pw + (2 * tt + kh)];
          const bf16 h = __float2bfloat16_rn(v);
          const bf16 l = __float2bfloat16_rn(v - __bfloat162float(h));
          hi[kh * 3 + kw] = __bfloat16_as_ushort(h);
          lo[kh * 3 + kw] = __bfloat16_as_ushort(l);
        }
      unsigned short row[kA0Cols];
#pragma unroll
      for (int q = 0; q < 9; ++q) row[q] = hi[q], row[9 + q] = lo[q];
      row[18] = row[19] = 0x3F80;  // bf16 1.0: the two halves of the bias
      row[20] = row[21] = row[22] = row[23] = 0;
#pragma unroll
      for (int j = 0; j < kA0Cols / 2; ++j) w[j] = static_cast<uint32_t>(row[2 * j]) | (static_cast<uint32_t>(row[2 * j + 1]) << 16);
    }
    const int vt1 = 2 * blk * kPackAlign + tt;  // row of the virtual sequence
    const int plane = (vt1 & 1) * 2 + pf;
    const long long r = (static_cast<long long>(plane) * Th + (vt1 >> 1)) * Fh + fh;
    uint4* dst = reinterpret_cast<uint4*>(a0 + r * kA0Cols);
    dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
    dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
    dst[2] = make_uint4(w[8], w[9], w[10], w[11]);
  }
}

// ------------------------------------------------------------------------------------------------ LayerNorm + scatter
// One warp per packed row; rows whose row_map entry is negative (gap rows) are skipped, the others are written to row
// row_map[r] of the dense result (the caller zero-fills it first).  Same arithmetic, in the same order, as
// layernorm_kernel (elementwise.cu), so the packed and the dense forward agree bit for bit.
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ void store4(float* p, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
__device__ __forceinline__ void store4(bf16* p, float a, float b, float c, float d) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&lo);
  u.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = u;
}

template <typename TOut>
__global__ void __launch_bounds__(256) layernorm_scatter_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                                const float* __restrict__ beta, TOut* __restrict__ out,
                                                                int rows, int d, const int32_t* __restrict__ row_map) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();
  if (row >= rows) return;
  const int dst = row_map[row];
  if (dst < 0) return;
  constexpr int kN = 8;  // d <= 1024
  const int nvec = d >> 2;
  const float inv_d = 1.0f / static_cast<float>(d);
  auto vidx = [&](int k) { return 64 * (k >> 1) + 2 * lane + (k & 1); };  // the lane -> column map of layernorm_kernel
  const float4* xr = reinterpret_cast<const float4*>(x + static_cast<long long>(row) * d);
  float4 v[kN];
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < kN; ++k)
    if (vidx(k) < nvec) {
      v[k] = __ldg(xr + vidx(k));
      s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    }
  const float mean = warp_sum(s) * inv_d;
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < kN; ++k)
    if (vidx(k) < nvec) {
      v[k].x -= mean, v[k].y -= mean, v[k].z -= mean, v[k].w -= mean;
      q += (v[k].x * v[k].x + v[k].y * v[k].y) + (v[k].z * v[k].z + v[k].w * v[k].w);
    }
  const float rstd = 1.0f / sqrtf(warp_sum(q) * inv_d + 1e-5f);
  TOut* orow = out + static_cast<long long>(dst) * d;
#pragma unroll
  for (int k = 0; k < kN; ++k) {
    const int i = vidx(k);
    if (i < nvec) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + i);
      const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + i);
      store4(orow + 4 * i, fmaf(v[k].x * rstd, g.x, b.x), fmaf(v[k].y * rstd, g.y, b.y), fmaf(v[k].z * rstd, g.z, b.z),
             fmaf(v[k].w * rstd, g.w, b.w));
    }
  }
}

}  // namespace

int launch_packed_plan(const long long* lengths, int B, int first, int step, int T, int T2, int n_rows, int n_tiles,
                       const PackedTables& tb, cudaStream_t st) {
  if (B <= 0) return 0;
  const size_t smem = static_cast<size_t>(4) * B * sizeof(int);
  if (smem > 48 * 1024) return -1;
  launch_pdl(packed_plan_kernel, dim3(1), dim3(kPlanThreads), smem, st, lengths, B, first, step, T, T2, n_rows, n_tiles, tb);
  return static_cast<int>(cudaGetLastError());
}

int launch_conv0_im2col_packed(const void* feats, bool feats_bf16, const long long* lengths, void* a0, int first, int step,
                               int F, int T, int T1, int F1, int Fh, int n_rows, const PackedTables& tb, cudaStream_t st) {
  if (n_rows <= 0) return 0;
  const size_t smem = static_cast<size_t>(F + 2) * (2 * kS1T + 2) * sizeof(float);
  const dim3 grid(n_rows / kPackAlign);
  if (feats_bf16)
    launch_pdl(conv0_im2col_packed_kernel<bf16>, grid, dim3(256), smem, st, reinterpret_cast<const bf16*>(feats), lengths,
               reinterpret_cast<bf16*>(a0), first, step, F, T, T1, F1, Fh, n_rows, tb);
  else
    launch_pdl(conv0_im2col_packed_kernel<float>, grid, dim3(256), smem, st, reinterpret_cast<const float*>(feats), lengths,
               reinterpret_cast<bf16*>(a0), first, step, F, T, T1, F1, Fh, n_rows, tb);
  return static_cast<int>(cudaGetLastError());
}

int launch_layernorm_scatter(const float* x, const float* gamma, const float* beta, void* out, bool out_bf16, int rows,
                             int d, const int32_t* row_map, cudaStream_t st) {
  if (rows <= 0) return 0;
  if (d % 4 != 0 || d > 1024) return -1;
  const int blocks = (rows + 7) / 8;
  if (out_bf16)
    launch_pdl(layernorm_scatter_kernel<bf16>, dim3(blocks), dim3(256), 0, st, x, gamma, beta, reinterpret_cast<bf16*>(out),
               rows, d, row_map);
  else
    launch_pdl(layernorm_scatter_kernel<float>, dim3(blocks), dim3(256), 0, st, x, gamma, beta,
               reinterpret_cast<float*>(out), rows, d, row_map);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace cfb
