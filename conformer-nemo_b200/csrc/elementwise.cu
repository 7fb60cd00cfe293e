// Memory-bound kernels of the encoder: LayerNorm, depth-wise time convolution (+ folded BatchNorm + Swish),
// the first 1->C strided convolution of the subsampling stack, the relative positional table, calc_length, and the
// validation path's im2col.  All are coalesced along the channel dimension with 128-bit accesses; reductions use
// warp shuffles; the depth-wise kernel stages its time halo in shared memory.
#include <cuda_fp16.h>

#include "common.cuh"

namespace cfb {
namespace {

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

__device__ __forceinline__ void store8(float* p, const float (&a)[8]) {
  store4(p, a[0], a[1], a[2], a[3]);
  store4(p + 4, a[4], a[5], a[6], a[7]);
}
__device__ __forceinline__ void store8(bf16* p, const float (&a)[8]) {  // one 16-byte store
  __nv_bfloat162 q0 = __floats2bfloat162_rn(a[0], a[1]), q1 = __floats2bfloat162_rn(a[2], a[3]);
  __nv_bfloat162 q2 = __floats2bfloat162_rn(a[4], a[5]), q3 = __floats2bfloat162_rn(a[6], a[7]);
  uint4 u;
  u.x = *reinterpret_cast<uint32_t*>(&q0);
  u.y = *reinterpret_cast<uint32_t*>(&q1);
  u.z = *reinterpret_cast<uint32_t*>(&q2);
  u.w = *reinterpret_cast<uint32_t*>(&q3);
  *reinterpret_cast<uint4*>(p) = u;
}

// ------------------------------------------------------------------------------------------------ LayerNorm
// One warp per row; the row lives in registers between the two reduction passes, so x is read from HBM exactly once.
// Statistics in fp32: mean, then the centred second moment (matches F.layer_norm).  NV = float4 per lane
// (d = 128*NV exactly) for the common widths; the generic instance (NV = 0) handles any d % 4 == 0 up to 1024.
constexpr int kMaxVec = 8;

template <typename TOut, int NV>
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, TOut* __restrict__ out,
                                                        int rows, int d, const int32_t* __restrict__ lens,
                                                        int frames_per_seq) {
  // Grid-stride over rows, one warp per row: the NEXT row's loads are issued before the current row is reduced, so a
  // warp always has a full row (2 KB at d = 512) in flight and blocks are not re-launched every eight rows.
  // A lane owns PAIRS of adjacent float4 (8 consecutive columns): 32-byte loads, one 16-byte store for bf16 outputs.
  const int warps_total = gridDim.x * (blockDim.x >> 5);
  int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();
  if (row >= rows) return;
  constexpr int kN = NV > 0 ? NV : kMaxVec;
  const int nvec = d >> 2;  // float4 per row
  const float inv_d = 1.0f / static_cast<float>(d);
  // float4 index of slot k: pair p = k / 2 covers float4 [64 p + 2 lane, 64 p + 2 lane + 1]
  auto vidx = [&](int k) { return 64 * (k >> 1) + 2 * lane + (k & 1); };
  float4 g[kN], b[kN];
#pragma unroll
  for (int k = 0; k < kN; ++k) {
    const int i = vidx(k);
    if (i < nvec) {
      g[k] = __ldg(reinterpret_cast<const float4*>(gamma) + i);
      b[k] = __ldg(reinterpret_cast<const float4*>(beta) + i);
    }
  }
  float4 nx[kN];
  auto fetch = [&](int r) {
    const float4* xr = reinterpret_cast<const float4*>(x + static_cast<long long>(r) * d);
#pragma unroll
    for (int k = 0; k < kN; ++k) {
      const int i = vidx(k);
      if (i < nvec) nx[k] = __ldg(xr + i);
    }
  };
  fetch(row);
  for (; row < rows; row += warps_total) {
    float4 v[kN];
#pragma unroll
    for (int k = 0; k < kN; ++k) v[k] = nx[k];
    if (row + warps_total < rows) fetch(row + warps_total);
    TOut* orow = out + static_cast<long long>(row) * d;
    if (lens != nullptr) {
      const int seq = row / frames_per_seq;
      if (row - seq * frames_per_seq >= lens[seq]) {
        for (int i = lane; i < nvec; i += 32) store4(orow + 4 * i, 0.f, 0.f, 0.f, 0.f);
        continue;
      }
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kN; ++k)
      if (vidx(k) < nvec) s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    const float mean = warp_sum(s) * inv_d;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < kN; ++k)
      if (vidx(k) < nvec) {
        v[k].x -= mean, v[k].y -= mean, v[k].z -= mean, v[k].w -= mean;
        q += (v[k].x * v[k].x + v[k].y * v[k].y) + (v[k].z * v[k].z + v[k].w * v[k].w);
      }
    const float rstd = 1.0f / sqrtf(warp_sum(q) * inv_d + 1e-5f);
#pragma unroll
    for (int k = 0; k < kN; k += 2) {
      const int i = vidx(k);
      float r8[8];
      r8[0] = fmaf(v[k].x * rstd, g[k].x, b[k].x), r8[1] = fmaf(v[k].y * rstd, g[k].y, b[k].y);
      r8[2] = fmaf(v[k].z * rstd, g[k].z, b[k].z), r8[3] = fmaf(v[k].w * rstd, g[k].w, b[k].w);
      if (k + 1 < kN) {
        r8[4] = fmaf(v[k + 1].x * rstd, g[k + 1].x, b[k + 1].x), r8[5] = fmaf(v[k + 1].y * rstd, g[k + 1].y, b[k + 1].y);
        r8[6] = fmaf(v[k + 1].z * rstd, g[k + 1].z, b[k + 1].z), r8[7] = fmaf(v[k + 1].w * rstd, g[k + 1].w, b[k + 1].w);
      }
      if (k + 1 < kN && i + 1 < nvec) {
        store8(orow + 4 * i, r8);
      } else if (i < nvec) {
        store4(orow + 4 * i, r8[0], r8[1], r8[2], r8[3]);
      }
    }
  }
}

// norm_out of one layer followed by norm_feed_forward1 of the next (conformer_modules.py:120 then :98 of the next
// layer) in one pass: y = LN1(x) is written back as the fp32 residual stream and LN2(y) as the bf16 GEMM operand.
// Saves one full read of the stream and one launch per layer.  Same one-warp-per-row scheme as layernorm_kernel.
// The first mean is taken of x - x[row][0] (exact for the elements within a factor 2 of the pivot): a residual stream
// with a large common offset keeps its fp32 accuracy, where the plain sum loses ~1e-3 at mean 1e3, std 0.1.
template <int NV>
__global__ void __launch_bounds__(256) layernorm_dual_kernel(const float* __restrict__ x, const float* __restrict__ g1,
                                                             const float* __restrict__ b1, float* __restrict__ out1,
                                                             const float* __restrict__ g2, const float* __restrict__ b2,
                                                             bf16* __restrict__ out2, int rows, int d) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();
  pdl_wait();
  if (row >= rows) return;
  constexpr int kN = NV > 0 ? NV : kMaxVec;
  const int nvec = d >> 2;
  const float4* xr = reinterpret_cast<const float4*>(x + static_cast<long long>(row) * d);
  const float pivot = __ldg(x + static_cast<long long>(row) * d);
  float4 v[kN];
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < kN; ++k) {
    const int i = lane + 32 * k;
    if (NV > 0 || i < nvec) {
      v[k] = __ldg(xr + i);
      v[k].x -= pivot, v[k].y -= pivot, v[k].z -= pivot, v[k].w -= pivot;
      s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    }
  }
  const float inv_d = 1.0f / static_cast<float>(d);
  float mean = warp_sum(s) * inv_d;
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < kN; ++k) {
    const int i = lane + 32 * k;
    if (NV > 0 || i < nvec) {
      v[k].x -= mean, v[k].y -= mean, v[k].z -= mean, v[k].w -= mean;
      q += (v[k].x * v[k].x + v[k].y * v[k].y) + (v[k].z * v[k].z + v[k].w * v[k].w);
    }
  }
  float rstd = 1.0f / sqrtf(warp_sum(q) * inv_d + 1e-5f);
  s = 0.f;
#pragma unroll
  for (int k = 0; k < kN; ++k) {
    const int i = lane + 32 * k;
    if (NV > 0 || i < nvec) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(g1) + i);
      const float4 b = __ldg(reinterpret_cast<const float4*>(b1) + i);
      v[k].x = fmaf(v[k].x * rstd, g.x, b.x), v[k].y = fmaf(v[k].y * rstd, g.y, b.y);
      v[k].z = fmaf(v[k].z * rstd, g.z, b.z), v[k].w = fmaf(v[k].w * rstd, g.w, b.w);
      store4(out1 + static_cast<long long>(row) * d + 4 * i, v[k].x, v[k].y, v[k].z, v[k].w);
      s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    }
  }
  mean = warp_sum(s) * inv_d;
  q = 0.f;
#pragma unroll
  for (int k = 0; k < kN; ++k) {
    const int i = lane + 32 * k;
    if (NV > 0 || i < nvec) {
      v[k].x -= mean, v[k].y -= mean, v[k].z -= mean, v[k].w -= mean;
      q += (v[k].x * v[k].x + v[k].y * v[k].y) + (v[k].z * v[k].z + v[k].w * v[k].w);
    }
  }
  rstd = 1.0f / sqrtf(warp_sum(q) * inv_d + 1e-5f);
#pragma unroll
  for (int k = 0; k < kN; ++k) {
    const int i = lane + 32 * k;
    if (NV > 0 || i < nvec) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(g2) + i);
      const float4 b = __ldg(reinterpret_cast<const float4*>(b2) + i);
      store4(out2 + static_cast<long long>(row) * d + 4 * i, fmaf(v[k].x * rstd, g.x, b.x), fmaf(v[k].y * rstd, g.y, b.y),
             fmaf(v[k].z * rstd, g.z, b.z), fmaf(v[k].w * rstd, g.w, b.w));
    }
  }
}

// ------------------------------------------------------------------------------------------------ depth-wise conv
// out[b,t,c] = swish(bias[c] + sum_k taps[k][c] * x[b, t + k - (K-1)/2, c]), zero outside [0,T); taps are (K, d).
// Block: 64 channels x 128 frames of one sequence.  The (128 + K - 1)-frame halo tile is staged in shared memory in
// the activation dtype with 16-byte cp.async copies (all in flight at once); each thread owns a channel pair and 16
// consecutive frames and slides the K-tap window over registers.  Reads and writes are 128-byte row segments.
constexpr int kDwC = 64, kDwT = 128, kDwMaxK = 31, kDwStrip = 16;

template <typename T>
__device__ __forceinline__ float2 load2(const T* p);
template <>
__device__ __forceinline__ float2 load2<float>(const float* p) {
  return *reinterpret_cast<const float2*>(p);
}
template <>
__device__ __forceinline__ float2 load2<bf16>(const bf16* p) {
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p));
}
__device__ __forceinline__ void store2(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
__device__ __forceinline__ void store2(bf16* p, float a, float b) {
  *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(a, b);
}

// d = a * b + c on two packed fp32 lanes (sm_100 FFMA2): the channel pair of a thread is one 64-bit register pair
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  unsigned long long ra, rb, rc, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}

template <typename T, bool kFast, int KS>  // KS > 0: compile-time tap count (31 in every shipped recipe); 0: runtime
__global__ void __launch_bounds__(256) depthwise_kernel(const T* __restrict__ x, const float* __restrict__ taps,
                                                        const float* __restrict__ bias, T* __restrict__ out, int T_len,
                                                        int d, int ksize_rt) {
  const int ksize = KS > 0 ? KS : ksize_rt;
  constexpr int kRows = kDwT + kDwMaxK - 1;
  constexpr int kVec = 16 / sizeof(T);       // elements per 16-byte chunk
  constexpr int kChunks = kDwC / kVec;       // chunks per tile row
  __shared__ __align__(16) T tile[kRows][kDwC];
  const int half = (ksize - 1) / 2;
  const int tblocks = (T_len + kDwT - 1) / kDwT;
  const int b = blockIdx.x / tblocks;
  const int t0 = (blockIdx.x % tblocks) * kDwT;
  const int c0 = blockIdx.y * kDwC;
  const T* xb = x + static_cast<long long>(b) * T_len * d;
  T* ob = out + static_cast<long long>(b) * T_len * d;
  const int span = kDwT + ksize - 1;
  static_assert((kChunks & (kChunks - 1)) == 0, "chunks per row must be a power of two");
  pdl_launch_dependents();
  pdl_wait();
  for (int i = threadIdx.x; i < span * kChunks; i += 256) {
    const int r = i / kChunks, ch = i & (kChunks - 1);
    const int t = t0 - half + r, c = c0 + ch * kVec;
    T* dst = &tile[r][ch * kVec];
    if (t >= 0 && t < T_len && c + kVec <= d) {
      const unsigned saddr = static_cast<unsigned>(__cvta_generic_to_shared(dst));
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(xb + static_cast<long long>(t) * d + c)
                   : "memory");
    } else {
#pragma unroll
      for (int e = 0; e < kVec; ++e) {
        const bool ok = t >= 0 && t < T_len && c + e < d;
        dst[e] = ok ? xb[static_cast<long long>(t) * d + c + e] : static_cast<T>(0.f);
      }
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  const int cp = threadIdx.x & 31;     // channel pair
  const int strip = threadIdx.x >> 5;  // 8 strips of 16 frames
  const int c = c0 + 2 * cp;
  const bool live = c < d;
  float2 w[kDwMaxK];
#pragma unroll
  for (int k = 0; k < kDwMaxK; ++k) {
    // taps are stored tap-major (ksize, d): a warp reads 256 contiguous bytes per tap
    w[k] = (live && k < ksize) ? __ldg(reinterpret_cast<const float2*>(taps + static_cast<long long>(k) * d + c))
                               : make_float2(0.f, 0.f);
  }
  const float b0 = live ? __ldg(bias + c) : 0.f, b1 = live ? __ldg(bias + c + 1) : 0.f;
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  if (!live) return;
  float2 acc[kDwStrip];
#pragma unroll
  for (int o = 0; o < kDwStrip; ++o) acc[o] = make_float2(b0, b1);
#pragma unroll
  for (int j = 0; j < kDwStrip + kDwMaxK - 1; ++j) {
    if (j < kDwStrip + ksize - 1) {
      const float2 vv = load2<T>(&tile[strip * kDwStrip + j][2 * cp]);
#pragma unroll
      for (int o = 0; o < kDwStrip; ++o) {
        const int k = j - o;
        if (k >= 0 && k < kDwMaxK) acc[o] = fma2(w[k], vv, acc[o]);
      }
    }
  }
#pragma unroll
  for (int o = 0; o < kDwStrip; ++o) {
    const int t = t0 + strip * kDwStrip + o;
    if (t < T_len) {
      float s0, s1;
      if constexpr (kFast) {  // swish(x) = h + h tanh(h), h = x/2
        const float h0 = 0.5f * acc[o].x, h1 = 0.5f * acc[o].y;
        float t0f, t1f;
        asm("tanh.approx.f32 %0, %1;" : "=f"(t0f) : "f"(h0));
        asm("tanh.approx.f32 %0, %1;" : "=f"(t1f) : "f"(h1));
        s0 = fmaf(h0, t0f, h0);
        s1 = fmaf(h1, t1f, h1);
      } else {
        s0 = acc[o].x / (1.f + expf(-acc[o].x));
        s1 = acc[o].y / (1.f + expf(-acc[o].y));
      }
      store2(ob + static_cast<long long>(t) * d + c, s0, s1);
    }
  }
}

// ------------------------------------------------------------------------------------------------ calc_length
// subsampling.py:272-282 evaluates floor((float(L) + 2p - k) / s + 1) in float32 per stage and truncates to int32;
// the same IEEE operations are issued here (no contraction) so the result is bit-identical for every int64 input.
__global__ void lengths_kernel(const long long* __restrict__ lengths, int32_t* __restrict__ out, int B, int T_full,
                               int n_stages) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  pdl_launch_dependents();
  pdl_wait();
  if (i >= B) return;
  if (lengths == nullptr) {
    float f = static_cast<float>(T_full);  // length=None: every row is T_full long (conformer_encoder.py:243-246)
    for (int s = 0; s < n_stages; ++s) f = floorf(__fadd_rn(__fdiv_rn(__fadd_rn(f, -1.0f), 2.0f), 1.0f));
    out[i] = static_cast<int32_t>(f);
    return;
  }
  float f = __ll2float_rn(lengths[i]);
  for (int s = 0; s < n_stages; ++s) f = floorf(__fadd_rn(__fdiv_rn(__fadd_rn(f, -1.0f), 2.0f), 1.0f));
  out[i] = static_cast<int32_t>(f);
}

// ------------------------------------------------------------------------------------------------ positional table
// row k <-> relative position (T-1-k); even columns sin(pos * div[m]), odd columns cos(pos * div[m])
// (multi_head_attention.py:235-248,292).  Accurate sinf/cosf: the argument reaches several thousand radians.
template <typename TOut>
__global__ void pos_table_kernel(TOut* __restrict__ out, const float* __restrict__ div_term, int T, int d) {
  const int k = blockIdx.x;
  pdl_launch_dependents();
  pdl_wait();
  const float pos = static_cast<float>(T - 1 - k);
  for (int m = threadIdx.x; m < d / 2; m += blockDim.x) {
    const float ang = __fmul_rn(pos, div_term[m]);
    store2(out + static_cast<long long>(k) * d + 2 * m, sinf(ang), cosf(ang));
  }
}

// ------------------------------------------------------------------------------------------------ first strided conv
// y1[b, t1, f1, c] = relu(bias[c] + sum_{kh,kw} w[c][kh][kw] * x[b][2 f1 + kw - 1][2 t1 + kh - 1])   (x is (B,F,T))
// written in the parity-split channels-last layout [B][plane = (t1&1)*2 + (f1&1)][Th][Fh][C] that lets the second
// convolution fetch each filter tap as one dense TMA box.  Positions with t1 >= T1 or f1 >= F1 are written as 0.
// Output-write bound (it is the largest tensor of the network): each thread keeps the 9 taps + bias of 8 channels in
// registers and walks over output positions; a warp's 16-byte stores cover 512 contiguous bytes.
constexpr int kS1T = 16;  // t1 rows per block
static_assert((kMaxFeatIn + 2) * (2 * kS1T + 2) * sizeof(float) <= 48 * 1024, "feature patch must fit the default shared memory");

template <typename TIn, typename TOut>
__global__ void __launch_bounds__(256) subsample_first_kernel(const TIn* __restrict__ feats,
                                                              const float* __restrict__ w9,
                                                              const float* __restrict__ bias, TOut* __restrict__ y,
                                                              int F, int T, int C, int T1, int F1, int Th, int Fh,
                                                              int groups_per_block) {
  extern __shared__ float patch[];  // [F + 2][2*kS1T + 2]: frames 2*t1_0 - 1 .. 2*(t1_0 + kS1T - 1) + 1
  const int pw = 2 * kS1T + 2;
  const int tblocks = (2 * Th + kS1T - 1) / kS1T;
  const int b = blockIdx.x / tblocks;
  const int t1_0 = (blockIdx.x % tblocks) * kS1T;
  const TIn* xb = feats + static_cast<long long>(b) * F * T;
  pdl_launch_dependents();
  pdl_wait();
  for (int i = threadIdx.x; i < (F + 2) * (2 * kS1T + 1); i += 256) {
    const int fr = i / (2 * kS1T + 1), tc = i % (2 * kS1T + 1);
    const int f = fr - 1, t = 2 * t1_0 - 1 + tc;
    float v = 0.f;
    if (f >= 0 && f < F && t >= 0 && t < T) v = static_cast<float>(xb[static_cast<long long>(f) * T + t]);
    patch[fr * pw + tc] = v;
  }
  __syncthreads();
  const int g_local = threadIdx.x % groups_per_block;
  const int lane_pos = threadIdx.x / groups_per_block;
  const int n_pos_lanes = 256 / groups_per_block;
  const int g = blockIdx.y * groups_per_block + g_local;  // 8 channels per group
  if (g * 8 >= C || lane_pos >= n_pos_lanes) return;
  // channel pairs share one FFMA2 (packed fp32): 36 instead of 72 multiply-adds per output position
  float2 w[4][9], bs[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    bs[j] = make_float2(__ldg(bias + g * 8 + 2 * j), __ldg(bias + g * 8 + 2 * j + 1));
#pragma unroll
    for (int q = 0; q < 9; ++q)
      w[j][q] = make_float2(__ldg(w9 + (g * 8 + 2 * j) * 9 + q), __ldg(w9 + (g * 8 + 2 * j + 1) * 9 + q));
  }
  const int positions = kS1T * 2 * Fh;
  for (int pos = lane_pos; pos < positions; pos += n_pos_lanes) {
    const int f1 = pos % (2 * Fh);
    const int tt = pos / (2 * Fh);
    const int t1 = t1_0 + tt;
    if (t1 >= 2 * Th) break;
    float acc[8];
    if ((t1 < T1) && (f1 < F1)) {
      float in[9];
#pragma unroll
      for (int kh = 0; kh < 3; ++kh)
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) in[kh * 3 + kw] = patch[(2 * f1 + kw) * pw + (2 * tt + kh)];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float2 a = bs[j];
#pragma unroll
        for (int q = 0; q < 9; ++q) a = fma2(w[j][q], make_float2(in[q], in[q]), a);
        acc[2 * j] = fmaxf(a.x, 0.f);
        acc[2 * j + 1] = fmaxf(a.y, 0.f);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    }
    const int plane = (t1 & 1) * 2 + (f1 & 1);
    const long long off =
        ((((static_cast<long long>(b) * 4 + plane) * Th + (t1 >> 1)) * Fh + (f1 >> 1)) * C) + g * 8;
    store8(y + off, acc);
  }
}

// ------------------------------------------------------------------------------------------------ conv 0 as a GEMM
// First strided convolution (1 -> C channels, 3x3, stride 2, pad 1; subsampling.py:99-105) on the tensor cores: this
// kernel gathers the 3x3 patch of every output position into one row of a bf16 matrix A0 whose row order IS the
// parity-split channels-last layout of y1 ([B][plane][Th][Fh]), and gemm_tc_kernel<EPI_RELU> multiplies it with the
// (C x 24) weight, writing y1 with its ordinary 2-D TMA stores.  Row = [x_hi (9) | x_lo (9) | 1 | 1 | 0 0 0 0]: the
// fp32 feature is split into two bf16 values (hi + lo carries 16 mantissa bits) and the bias rides on the two
// constant columns the same way, so only the nine weights are rounded to bf16.  Rows of positions outside (T1, F1)
// -- the padding of the planes -- are all zero, which makes relu(0) = 0 exactly what the second conv must see.
constexpr int kA0Cols = 24;
template <typename TIn>
__global__ void __launch_bounds__(256) conv0_im2col_kernel(const TIn* __restrict__ feats, bf16* __restrict__ a0, int F,
                                                           int T, int T1, int F1, int Th, int Fh) {
  extern __shared__ float patch[];  // [F + 2][2*kS1T + 2]: frames 2*t1_0 - 1 .. 2*(t1_0 + kS1T - 1) + 1
  const int pw = 2 * kS1T + 2;
  const int tblocks = (2 * Th + kS1T - 1) / kS1T;
  const int b = blockIdx.x / tblocks;
  const int t1_0 = (blockIdx.x % tblocks) * kS1T;
  const TIn* xb = feats + static_cast<long long>(b) * F * T;
  pdl_launch_dependents();
  pdl_wait();
  for (int i = threadIdx.x; i < (F + 2) * (2 * kS1T + 1); i += 256) {
    const int fr = i / (2 * kS1T + 1), tc = i % (2 * kS1T + 1);
    const int f = fr - 1, t = 2 * t1_0 - 1 + tc;
    float v = 0.f;
    if (f >= 0 && f < F && t >= 0 && t < T) v = static_cast<float>(xb[static_cast<long long>(f) * T + t]);
    patch[fr * pw + tc] = v;
  }
  __syncthreads();
  const int positions = kS1T * 2 * Fh;
  for (int pos = threadIdx.x; pos < positions; pos += 256) {
    // consecutive threads -> consecutive rows of one plane (same f1 parity), then the other parity, then the next t1
    const int fh = pos % Fh;
    const int pf = (pos / Fh) & 1;
    const int tt = pos / (2 * Fh);
    const int f1 = 2 * fh + pf;
    const int t1 = t1_0 + tt;
    if (t1 >= 2 * Th) break;
    uint32_t w[kA0Cols / 2];
#pragma unroll
    for (int j = 0; j < kA0Cols / 2; ++j) w[j] = 0u;
    if (t1 < T1 && f1 < F1) {
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
    const int plane = (t1 & 1) * 2 + pf;
    const long long r = ((static_cast<long long>(b) * 4 + plane) * Th + (t1 >> 1)) * Fh + fh;
    uint4* dst = reinterpret_cast<uint4*>(a0 + r * kA0Cols);
    dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
    dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
    dst[2] = make_uint4(w[8], w[9], w[10], w[11]);
  }
}

// ------------------------------------------------------------------------------------------------ im2col (validation)
__global__ void im2col_kernel(const float* __restrict__ y, float* __restrict__ cols, int B, int C, int Th, int Fh,
                              int To, int Fo) {
  const long long total = static_cast<long long>(B) * To * Fo * 9 * C;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    long long r = i / C;
    const int tap = static_cast<int>(r % 9);
    r /= 9;
    const int fo = static_cast<int>(r % Fo);
    r /= Fo;
    const int to = static_cast<int>(r % To);
    const int b = static_cast<int>(r / To);
    const int kh = tap / 3, kw = tap % 3;
    const int t1 = 2 * to + kh - 1, f1 = 2 * fo + kw - 1;
    float v = 0.f;
    if (t1 >= 0 && t1 < 2 * Th && f1 >= 0 && f1 < 2 * Fh) {
      const int plane = (t1 & 1) * 2 + (f1 & 1);
      v = y[((((static_cast<long long>(b) * 4 + plane) * Th + (t1 >> 1)) * Fh + (f1 >> 1)) * C) + c];
    }
    cols[i] = v;
  }
}

// ------------------------------------------------------------------------------------------------ bf16 -> fp16
// eight elements per thread (cols % 8 == 0); element-wise, so dst may alias src when both are dense
__global__ void __launch_bounds__(256) bf16_to_f16_kernel(const bf16* src, long long ld, __half* dst, long long rows, int cols) {
  const int c8 = cols >> 3;
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  pdl_launch_dependents();
  pdl_wait();
  if (i >= rows * c8) return;
  const long long r = i / c8;
  const int c = static_cast<int>(i - r * c8) * 8;
  const uint4 u = *reinterpret_cast<const uint4*>(src + r * ld + c);
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
  uint32_t o[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[k]));
    const __half2 hh = __floats2half2_rn(f.x, f.y);
    o[k] = *reinterpret_cast<const uint32_t*>(&hh);
  }
  *reinterpret_cast<uint4*>(dst + r * cols + c) = make_uint4(o[0], o[1], o[2], o[3]);
}

}  // namespace
int launch_bf16_to_f16(const void* src, long long ld, void* dst, long long rows, int cols, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return 0;
  if (cols % 8 != 0 || ld % 8 != 0) return -1;
  const long long n = rows * (cols >> 3);
  launch_pdl(bf16_to_f16_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, st,
             reinterpret_cast<const bf16*>(src), ld, reinterpret_cast<__half*>(dst), rows, cols);
  return static_cast<int>(cudaGetLastError());
}


int launch_layernorm(const float* x, const float* gamma, const float* beta, void* out, bool out_bf16, int rows, int d,
                     const int32_t* lens, int frames_per_seq, cudaStream_t st) {
  if (rows <= 0) return 0;
  if (d % 4 != 0 || d > 128 * kMaxVec) return -1;
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  int blocks = (rows + 7) / 8;
  if (blocks > 2 * sms) blocks = 2 * sms;  // two resident CTAs per SM (90 registers): one balanced wave, each warp looping over rows
#define CFB_LN(T, NV)                                                                                            \
  launch_pdl(layernorm_kernel<T, NV>, dim3(blocks), dim3(256), 0, st, x, gamma, beta, reinterpret_cast<T*>(out), rows, \
             d, lens, frames_per_seq)
  if (out_bf16) {
    if (d == 512) CFB_LN(bf16, 4);
    else if (d == 256) CFB_LN(bf16, 2);
    else CFB_LN(bf16, 0);
  } else {
    if (d == 512) CFB_LN(float, 4);
    else if (d == 256) CFB_LN(float, 2);
    else CFB_LN(float, 0);
  }
#undef CFB_LN
  return static_cast<int>(cudaGetLastError());
}

int launch_layernorm_dual(const float* x, const float* g1, const float* b1, float* out1, const float* g2, const float* b2,
                          void* out2_bf16, int rows, int d, cudaStream_t st) {
  if (rows <= 0) return 0;
  if (d % 4 != 0 || d > 128 * kMaxVec) return -1;
  const int blocks = (rows + 7) / 8;
  bf16* o2 = reinterpret_cast<bf16*>(out2_bf16);
  if (d == 512) launch_pdl(layernorm_dual_kernel<4>, dim3(blocks), dim3(256), 0, st, x, g1, b1, out1, g2, b2, o2, rows, d);
  else if (d == 256) launch_pdl(layernorm_dual_kernel<2>, dim3(blocks), dim3(256), 0, st, x, g1, b1, out1, g2, b2, o2, rows, d);
  else launch_pdl(layernorm_dual_kernel<0>, dim3(blocks), dim3(256), 0, st, x, g1, b1, out1, g2, b2, o2, rows, d);
  return static_cast<int>(cudaGetLastError());
}

int launch_depthwise(const void* x, const float* taps, const float* bias, void* out, bool is_bf16, int B, int T, int d,
                     int ksize, cudaStream_t st) {
  if (B <= 0 || T <= 0) return 0;
  if (ksize > kDwMaxK || (ksize & 1) == 0 || d % 2 != 0) return -1;
  dim3 grid(B * ((T + kDwT - 1) / kDwT), (d + kDwC - 1) / kDwC);
  if (is_bf16) {
    if (ksize == 31)
      launch_pdl(depthwise_kernel<bf16, true, 31>, grid, dim3(256), 0, st, reinterpret_cast<const bf16*>(x), taps, bias,
                 reinterpret_cast<bf16*>(out), T, d, ksize);
    else
      launch_pdl(depthwise_kernel<bf16, true, 0>, grid, dim3(256), 0, st, reinterpret_cast<const bf16*>(x), taps, bias,
                 reinterpret_cast<bf16*>(out), T, d, ksize);
  } else {
    depthwise_kernel<float, false, 0><<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(x), taps, bias,
                                                            reinterpret_cast<float*>(out), T, d, ksize);
  }
  return static_cast<int>(cudaGetLastError());
}

int launch_lengths(const long long* lengths, int32_t* out, int B, int T_full, int n_stages, cudaStream_t st) {
  if (B <= 0) return 0;
  launch_pdl(lengths_kernel, dim3((B + 127) / 128), dim3(128), 0, st, lengths, out, B, T_full, n_stages);
  return static_cast<int>(cudaGetLastError());
}

int launch_pos_table(void* out, bool out_bf16, const float* div_term, int T, int d, cudaStream_t st) {
  if (T <= 0) return 0;
  if (out_bf16)
    launch_pdl(pos_table_kernel<bf16>, dim3(2 * T - 1), dim3(128), 0, st, reinterpret_cast<bf16*>(out), div_term, T, d);
  else
    pos_table_kernel<float><<<2 * T - 1, 128, 0, st>>>(reinterpret_cast<float*>(out), div_term, T, d);
  return static_cast<int>(cudaGetLastError());
}

int launch_subsample_first(const void* feats, bool feats_bf16, const float* w9, const float* bias, void* y_out,
                           bool out_bf16, int B, int F, int T, int C, int T1, int F1, int Th, int Fh, cudaStream_t st) {
  if (B <= 0) return 0;
  if (C % 8 != 0) return -1;
  const int tblocks = (2 * Th + kS1T - 1) / kS1T;
  const size_t smem = static_cast<size_t>(F + 2) * (2 * kS1T + 2) * sizeof(float);
  const int groups = C / 8;
  const int gpb = groups < 64 ? groups : 64;  // channel groups per block; the other threads walk positions
  const dim3 grid(B * tblocks, (groups + gpb - 1) / gpb);
#define CFB_S1(TIN, TOUT)                                                                                         \
  launch_pdl(subsample_first_kernel<TIN, TOUT>, grid, dim3(256), smem, st, reinterpret_cast<const TIN*>(feats), w9,  \
             bias, reinterpret_cast<TOUT*>(y_out), F, T, C, T1, F1, Th, Fh, gpb)
  if (feats_bf16) {
    if (out_bf16)
      CFB_S1(bf16, bf16);
    else
      CFB_S1(bf16, float);
  } else {
    if (out_bf16)
      CFB_S1(float, bf16);
    else
      CFB_S1(float, float);
  }
#undef CFB_S1
  return static_cast<int>(cudaGetLastError());
}

int launch_conv0_im2col(const void* feats, bool feats_bf16, void* a0, int B, int F, int T, int T1, int F1, int Th, int Fh,
                        cudaStream_t st) {
  if (B <= 0) return 0;
  const int tblocks = (2 * Th + kS1T - 1) / kS1T;
  const size_t smem = static_cast<size_t>(F + 2) * (2 * kS1T + 2) * sizeof(float);
  if (feats_bf16)
    launch_pdl(conv0_im2col_kernel<bf16>, dim3(B * tblocks), dim3(256), smem, st, reinterpret_cast<const bf16*>(feats),
               reinterpret_cast<bf16*>(a0), F, T, T1, F1, Th, Fh);
  else
    launch_pdl(conv0_im2col_kernel<float>, dim3(B * tblocks), dim3(256), smem, st, reinterpret_cast<const float*>(feats),
               reinterpret_cast<bf16*>(a0), F, T, T1, F1, Th, Fh);
  return static_cast<int>(cudaGetLastError());
}

int launch_im2col(const float* y_in, float* cols, int B, int C, int Th, int Fh, int To, int Fo, cudaStream_t st) {
  const long long total = static_cast<long long>(B) * To * Fo * 9 * C;
  if (total <= 0) return 0;
  const int blocks = static_cast<int>(total / 256 + 1 < 65535 * 8 ? total / 256 + 1 : 65535 * 8);
  im2col_kernel<<<blocks, 256, 0, st>>>(y_in, cols, B, C, Th, Fh, To, Fo);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace cfb
