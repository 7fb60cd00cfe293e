// Helpers shared by the transducer decode kernels (rnnt_greedy.cu, rnnt_beam.cu): the fence-free grid barrier of a
// cooperative launch, small dot-product / activation helpers, the packed (value, index) arg-max key, the row partition
// over CTAs and the load of a CTA's rows into shared memory, and the host side both entry points share: weight
// validation, the device query and the joint.enc projection (defined in rnnt_greedy.cu).
#pragma once

#include "../../include/cfb.h"
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

// The rows of the row partition a CTA keeps in shared memory for the whole decode (P: the kernel's parameters):
//   s_wl [nu][4][2H]  the LSTM rows of hidden units [u_lo, u_lo + nu), gate-major per unit: [w_ih row | w_hh row],
//   s_bl [nu][4]      their b_ih + b_hh,
//   s_wp [np][H]      joint.pred rows [p_lo, p_lo + np),
//   s_wj [nj][J]      output-layer rows [j_lo, j_lo + nj).
template <class P>
__device__ __forceinline__ void load_row_weights(const P& p, int u_lo, int nu, int p_lo, int np, int j_lo, int nj, float* s_wl,
                                                 float* s_bl, float* s_wp, float* s_wj) {
  const int H = p.H, J = p.J, tid = threadIdx.x, nt = blockDim.x;
  for (int i = tid; i < nu * 4 * (2 * H / 4); i += nt) {
    const int k4 = i % (2 * H / 4), r = i / (2 * H / 4), gate = r & 3, ul = r >> 2;
    const int row = gate * H + u_lo + ul;
    const float* src = k4 < H / 4 ? p.w_ih + static_cast<size_t>(row) * H + k4 * 4
                                  : p.w_hh + static_cast<size_t>(row) * H + (k4 - H / 4) * 4;
    reinterpret_cast<float4*>(s_wl)[i] = __ldg(reinterpret_cast<const float4*>(src));
  }
  for (int i = tid; i < nu * 4; i += nt) {
    const int row = (i & 3) * H + u_lo + (i >> 2);
    s_bl[i] = p.b_ih[row] + p.b_hh[row];
  }
  for (int i = tid; i < np * (H / 4); i += nt)
    reinterpret_cast<float4*>(s_wp)[i] = __ldg(reinterpret_cast<const float4*>(p.w_pred + static_cast<size_t>(p_lo) * H) + i);
  for (int i = tid; i < nj * (J / 4); i += nt)
    reinterpret_cast<float4*>(s_wj)[i] = __ldg(reinterpret_cast<const float4*>(p.w_out + static_cast<size_t>(j_lo) * J) + i);
}

inline size_t align256(size_t v) { return (v + 255) / 256 * 256; }

}  // namespace

// ---- host side of cfb_op_rnnt_greedy / cfb_op_rnnt_beam ------------------------------------------------------------------

// The sizes, activation, pointers and encoder-output dtype both decoders accept.
bool rnnt_weights_valid(const cfb_rnnt_weights& w, int x_dtype);

// SMs and opt-in shared memory per block of the current device: CFB_ERR_CUDA, CFB_ERR_UNSUPPORTED without cooperative launch.
int rnnt_device_query(int* sms, int* max_smem);

// The joint.enc buffers at the end of both scratch layouts, from `off` on: encp (B*T, J) fp32 = joint.enc(encoded) and
// the split operands of its GEMM, a (B*T, 3E) and w (J, 3E) bf16.
struct RnntEncScratch {
  size_t encp_off, a_off, w_off, end;
};
inline RnntEncScratch rnnt_enc_scratch(size_t off, int E, int J, int B, int T) {
  RnntEncScratch s;
  s.encp_off = off;
  off += align256(sizeof(float) * static_cast<size_t>(B) * T * J);
  s.a_off = off;
  off += align256(sizeof(bf16) * static_cast<size_t>(B) * T * 3 * E);
  s.w_off = off;
  off += align256(sizeof(bf16) * static_cast<size_t>(J) * 3 * E);
  s.end = off;
  return s;
}

// Enqueues encp = encoded W_enc^T + b_enc over every frame into the scratch at `ws` (0 or CFB_ERR_CUDA).
int rnnt_joint_enc(const cfb_rnnt_weights& w, const void* encoded, int x_dtype, int B, int T, uint8_t* ws, const RnntEncScratch& s,
                   cudaStream_t st);

}  // namespace cfb
