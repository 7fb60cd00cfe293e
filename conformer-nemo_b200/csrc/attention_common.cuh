// Device helpers shared by the tensor-core attention kernels (attention_tc.cu, attention_tcp.cu, attention_tc128.cu).
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

namespace cfb {
namespace attn {

// (q + v) enters the fp16 G MMA (the position term, fp16 operands and fp16 accumulator) divided by kGScale, a power of
// two, for headroom in the accumulator; the window is multiplied back where it is added to the scores
constexpr float kGScale = 16.f, kGScaleInv = 1.f / 16.f;
constexpr uint16_t kGScaleH = 0x4C00;  // kGScale as fp16

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  __half2 t = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}
__device__ __forceinline__ float4 lds_f32x4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}

// 32 consecutive words from shared memory in one asm statement (see ptx::lds_f32x32)
__device__ __forceinline__ void lds_u32x32(uint32_t addr, uint32_t (&v)[32]) {
  asm volatile(
      "ld.shared.b32 %0, [%32+0];\n ld.shared.b32 %1, [%32+4];\n ld.shared.b32 %2, [%32+8];\n ld.shared.b32 %3, [%32+12];\n"
      "ld.shared.b32 %4, [%32+16];\n ld.shared.b32 %5, [%32+20];\n ld.shared.b32 %6, [%32+24];\n ld.shared.b32 %7, [%32+28];\n"
      "ld.shared.b32 %8, [%32+32];\n ld.shared.b32 %9, [%32+36];\n ld.shared.b32 %10, [%32+40];\n ld.shared.b32 %11, [%32+44];\n"
      "ld.shared.b32 %12, [%32+48];\n ld.shared.b32 %13, [%32+52];\n ld.shared.b32 %14, [%32+56];\n ld.shared.b32 %15, [%32+60];\n"
      "ld.shared.b32 %16, [%32+64];\n ld.shared.b32 %17, [%32+68];\n ld.shared.b32 %18, [%32+72];\n ld.shared.b32 %19, [%32+76];\n"
      "ld.shared.b32 %20, [%32+80];\n ld.shared.b32 %21, [%32+84];\n ld.shared.b32 %22, [%32+88];\n ld.shared.b32 %23, [%32+92];\n"
      "ld.shared.b32 %24, [%32+96];\n ld.shared.b32 %25, [%32+100];\n ld.shared.b32 %26, [%32+104];\n ld.shared.b32 %27, [%32+108];\n"
      "ld.shared.b32 %28, [%32+112];\n ld.shared.b32 %29, [%32+116];\n ld.shared.b32 %30, [%32+120];\n ld.shared.b32 %31, [%32+124];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
        "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(addr)
      : "memory");
}
// kind::f16 instruction descriptor with fp16 A / B and an fp16 accumulator (tools/ubench_f16acc.cu: bf16 operands with an
// fp16 accumulator are an illegal instruction; an fp16 accumulator takes one 32-bit TMEM column per element)
__host__ __device__ constexpr uint32_t make_idesc_f16_f16acc(int m, int n) {
  return (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

}  // namespace attn
}  // namespace cfb
