// Helpers shared by the transducer decode kernels (rnnt_greedy.cu, rnnt_beam.cu): the fence-free grid barrier of a
// cooperative launch, small dot-product / activation helpers, the packed (value, index) arg-max key, the row partition
// over CTAs and the split-operand conversion that feeds joint.enc to the tcgen05 GEMM.
#pragma once

#include "common.cuh"

namespace cfb {
namespace {

__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Grid barrier (all CTAs are co-resident: cooperative launch).  counter[0] counts arrivals (monotonic), counter[64]
// (another 128-byte line) is the release flag the last arriver publishes, so the spinning CTAs poll a line no atomic hits.
__device__ __forceinline__ void grid_sync(unsigned int* counter, unsigned int& target) {
  // Release/acquire chain instead of two full fences: bar.sync orders the CTA's writes before thread 0's acq_rel
  // arrival (cumulative), the last arriver publishes the flag with a release store, pollers acquire it, bar.sync hands
  // the ordering to the rest of the CTA.  Every mutable global datum is read with ld.global.cg (never from L1).
  target += gridDim.x;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int old;
    asm volatile("atom.add.acq_rel.gpu.global.u32 %0, [%1], 1;" : "=r"(old) : "l"(counter) : "memory");
    if (old + 1u == target) {
      asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(counter + 64), "r"(target) : "memory");
    } else {
      while (ld_acquire_u32(counter + 64) < target) {
      }
    }
  }
  __syncthreads();
}

__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float dot4(const float4 a, const float4 b, float acc) {
  acc = fmaf(a.x, b.x, acc);
  acc = fmaf(a.y, b.y, acc);
  acc = fmaf(a.z, b.z, acc);
  return fmaf(a.w, b.w, acc);
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }
__device__ __forceinline__ float act_fn(float x, int act) {
  return act == 0 ? fmaxf(x, 0.f) : (act == 1 ? sigmoidf_(x) : tanhf(x));
}
__device__ __forceinline__ unsigned long long pack_key(float v, int idx) {
  unsigned int u = __float_as_uint(v);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return (static_cast<unsigned long long>(u) << 32) | static_cast<unsigned long long>(0xffffffffu - static_cast<unsigned int>(idx));
}
__device__ __forceinline__ void unpack_key(unsigned long long key, float* v, int* idx) {
  unsigned int u = static_cast<unsigned int>(key >> 32);
  u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  *v = __uint_as_float(u);
  *idx = static_cast<int>(0xffffffffu - static_cast<unsigned int>(key & 0xffffffffu));
}

// rows [lo, hi) of `n` rows owned by CTA c of g
__device__ __forceinline__ void row_range(int n, int c, int g, int* lo, int* hi) {
  *lo = static_cast<int>(static_cast<long long>(n) * c / g);
  *hi = static_cast<int>(static_cast<long long>(n) * (c + 1) / g);
}

// fp32 (rows, K) -> bf16 (rows, 3K) [hi | hi | lo]   (mode 0, activations)
//                -> bf16 (rows, 3K) [hi | lo | hi]   (mode 1, weights)
// bf16 input (mode 2): (rows, K) -> (rows, 2K) [x | x]
__global__ void __launch_bounds__(256) split_bf16_kernel(const void* __restrict__ x, bf16* __restrict__ y, long long rows, int K,
                                                         int mode) {
  const long long n = rows * K;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / K;
    const int k = static_cast<int>(i % K);
    if (mode == 2) {
      const bf16 v = reinterpret_cast<const bf16*>(x)[i];
      y[r * 2 * K + k] = v;
      y[r * 2 * K + K + k] = v;
    } else {
      const float v = reinterpret_cast<const float*>(x)[i];
      const bf16 hi = __float2bfloat16_rn(v);
      const bf16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
      bf16* o = y + r * 3 * K;
      o[k] = hi;
      o[K + k] = mode == 0 ? hi : lo;
      o[2 * K + k] = mode == 0 ? lo : hi;
    }
  }
}

inline size_t align256(size_t v) { return (v + 255) / 256 * 256; }

}  // namespace
}  // namespace cfb
