// Tail of the Conformer convolution module in ONE kernel (conformer_modules.py:168-180):
//
//   c = swish(BN(depthwise_conv(g)))      k = 31 taps along time, eval BatchNorm folded into taps + bias
//   x += pointwise_conv2(c) + b2          1x1 conv = GEMM over channels, residual update of the fp32 stream
//
// The stand-alone version writes c (N x d bf16) to HBM and reads it back as the A operand of a tcgen05 GEMM.  Here the
// depth-wise output never leaves the SM: one CTA owns 128 frames of one sequence and ALL d output channels
// (accumulator = 128 lanes x d <= 512 TMEM columns).  Per 64-channel k-block
//   warp 0      TMA: the (128 + 30) x 64 halo tile of g (3-D map over (d, T, B): frames outside the sequence are
//               zero-filled by the hardware = the conv's zero padding) and the 32 x 64 fp32 tap/bias block, 3 stages
//   warp 2      TMA: the pointwise weight boxes (SW128, 3-slot ring)
//   warps 3..18 depth-wise producers, two groups of eight that take alternate k-blocks (four warps per scheduler keep
//               the FMA pipe fed): thread = (channel pair, 16-frame strip), sliding 31-tap window in registers with
//               packed FFMA2, Swish, bf16 pack, stored straight into the 128-byte-swizzled K-major A tile that the
//               UMMA descriptor expects (row = frame, 16-byte chunk index XOR row & 7), fence.proxy.async + mbarrier
//   warp 1      tcgen05.mma issuer: A (SIMT-written smem) x W^T (TMA-written smem) -> TMEM, N split in <= 256 columns
// and after the last k-block the same sixteen warps run the epilogue: tcgen05.ld, + b2, swizzled staging boxes,
// cp.reduce.async.bulk (.add.f32) into x with TMA clipping at the end of the sequence.
// Arithmetic order is the stand-alone kernels' (taps ascending, k-blocks ascending): results are bit-identical to
// depthwise_kernel + gemm_tc_kernel<EPI_RESID>.
#include <stdio.h>

#include "common.cuh"
#include "ptx.cuh"

namespace cfb {

namespace {

constexpr int kTileT = 128;                  // frames per CTA
constexpr int kTaps = 31;
constexpr int kHalo = (kTaps - 1) / 2;
constexpr int kGRows = kTileT + kTaps - 1;   // 158 input frames per tile
constexpr int kKC = 64;                      // channels per k-block (one 128-byte swizzle row of bf16)
constexpr int kStrip = 16;                   // frames per producer thread
constexpr int kStripWarps = kTileT / kStrip; // 8 warps cover the 128 frames of one k-block
constexpr int kGroups = 2;                   // producer groups: group q computes the k-blocks kb = q (mod 2)
constexpr int kProdWarps = kGroups * kStripWarps;
constexpr int kCtrlWarps = 3;                  // g/taps loader, MMA issuer, weight loader
constexpr int kThreads = 32 * (kCtrlWarps + kProdWarps);
constexpr int kWStages = 3;
constexpr int kWStage = 256 * 128;           // one pointwise-weight box: <= 256 output channels x 64 k
constexpr int kAStage = kTileT * 128;
constexpr int kGStages = 3;
constexpr int kGBytes = kGRows * 128;
constexpr int kGStage = 20 * 1024;
constexpr int kTapBytes = 32 * kKC * 4;
constexpr int kOffW = 0;
constexpr int kOffA = kOffW + kWStages * kWStage;
constexpr int kOffG = kOffA + 2 * kAStage;
constexpr int kOffT = kOffG + kGStages * kGStage;
constexpr int kOffBias = kOffT + kGStages * kTapBytes;  // float[512]: pointwise_conv2 bias
constexpr int kOffBar = kOffBias + 2048;
constexpr int kSmemNeeded = kOffBar + 256;
constexpr int kSmemTotal = kSmemNeeded + 1024;
static_assert(kSmemTotal <= 227 * 1024, "shared memory budget");
static_assert(kGBytes <= kGStage, "halo tile stage");
static_assert(kProdWarps * 2 * 4096 <= kOffG, "epilogue staging reuses the weight ring and the A tiles");

struct DwPwParams {
  int T, d, num_kb, nc, bnc, tblocks;
  uint32_t tmem_cols;
  const float* bias2;
};

__device__ __forceinline__ float2 lds64f(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t lds32u(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts32u(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
// d = a * b + c on two packed fp32 lanes (FFMA2)
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  unsigned long long ra, rb, rc, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}
__device__ __forceinline__ float swish_fast(float v) {  // swish(v) = h + h tanh(h), h = v / 2 (as depthwise_kernel)
  const float h = 0.5f * v;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

__global__ void __launch_bounds__(kThreads, 1)
dw_pw_kernel(const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmT,
             const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmO, const DwPwParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  if (static_cast<int>(smem - smem_raw) + kSmemNeeded > kSmemTotal) __trap();
  const uint32_t sbase = ptx::smem_u32(smem);
  // barriers (8 bytes each): g_full[3] g_empty[3] a_full[2] a_empty[2] w_full[3] w_empty[3] acc_full
  const uint32_t bar0 = sbase + kOffBar;
  const uint32_t g_full = bar0, g_empty = bar0 + 24, a_full = bar0 + 48, a_empty = bar0 + 64;
  const uint32_t w_full = bar0 + 80, w_empty = bar0 + 104, acc_full = bar0 + 128;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffBar + 136);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x / p.tblocks;
  const int t0 = (blockIdx.x - b * p.tblocks) * kTileT;

  if (warp == 0) {
    if (lane == 0) {
      ptx::prefetch_tmap(&tmG);
      ptx::prefetch_tmap(&tmT);
      ptx::prefetch_tmap(&tmW);
      ptx::prefetch_tmap(&tmO);
      for (int s = 0; s < kGStages; ++s) {
        ptx::mbar_init_a(g_full + 8 * s, 1);
        ptx::mbar_init_a(g_empty + 8 * s, kStripWarps);
      }
      for (int s = 0; s < 2; ++s) {
        ptx::mbar_init_a(a_full + 8 * s, kStripWarps);
        ptx::mbar_init_a(a_empty + 8 * s, 1);
      }
      for (int s = 0; s < kWStages; ++s) {
        ptx::mbar_init_a(w_full + 8 * s, 1);
        ptx::mbar_init_a(w_empty + 8 * s, 1);
      }
      ptx::mbar_init_a(acc_full, 1);
      ptx::fence_mbar_init();
    }
    __syncwarp();
    ptx::tmem_alloc(tmem_slot, p.tmem_cols);
  } else if (warp >= kCtrlWarps) {
    // pointwise_conv2 bias -> shared memory (a weight: not produced by the previous kernel, safe before pdl_wait)
    float* bias_s = reinterpret_cast<float*>(smem + kOffBias);
    for (int i = static_cast<int>(threadIdx.x) - 32 * kCtrlWarps; i < p.d; i += 32 * kProdWarps) bias_s[i] = __ldg(p.bias2 + i);
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer: halo tiles of g + tap blocks
    if (lane == 0) {
      int gs = 0;
      uint32_t gphase = 0;
      for (int kb = 0; kb < p.num_kb; ++kb) {
        ptx::mbar_wait_a(g_empty + 8 * gs, gphase ^ 1);
        ptx::mbar_arrive_expect_tx_a(g_full + 8 * gs, kGBytes + kTapBytes);
        ptx::tma_load_3d(smem + kOffG + gs * kGStage, &tmG, reinterpret_cast<uint64_t*>(smem + kOffBar + 8 * gs),
                         kb * kKC, t0 - kHalo, b);
        ptx::tma_load_2d(smem + kOffT + gs * kTapBytes, &tmT, reinterpret_cast<uint64_t*>(smem + kOffBar + 8 * gs),
                         kb * kKC, 0);
        if (++gs == kGStages) {
          gs = 0;
          gphase ^= 1;
        }
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------------ TMA producer: pointwise weight boxes
    // (its own warp: a w_empty wait -- which needs MMAs, hence finished A tiles -- must never delay a halo prefetch)
    if (lane == 0) {
      int wslot = 0;
      uint32_t wphase = 0;
      for (int kb = 0; kb < p.num_kb; ++kb) {
        for (int nh = 0; nh < p.nc; ++nh) {
          ptx::mbar_wait_a(w_empty + 8 * wslot, wphase ^ 1);
          ptx::mbar_arrive_expect_tx_a(w_full + 8 * wslot, static_cast<uint32_t>(p.bnc) * 128u);
          ptx::tma_load_2d(smem + kOffW + wslot * kWStage, &tmW,
                           reinterpret_cast<uint64_t*>(smem + kOffBar + 80 + 8 * wslot), kb * kKC, nh * p.bnc);
          if (++wslot == kWStages) {
            wslot = 0;
            wphase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      const uint32_t idesc = ptx::make_idesc_bf16(kTileT, p.bnc, 0, 0);
      int wslot = 0;
      uint32_t wphase = 0;
      for (int kb = 0; kb < p.num_kb; ++kb) {
        const int s = kb & 1;
        ptx::mbar_wait_a(a_full + 8 * s, (kb >> 1) & 1);
        ptx::tc_fence_after();
        const uint64_t da = ptx::make_sdesc_sw128(sbase + kOffA + s * kAStage, 16, 1024);
        for (int nh = 0; nh < p.nc; ++nh) {
          ptx::mbar_wait_a(w_full + 8 * wslot, wphase);
          ptx::tc_fence_after();
          const uint64_t db = ptx::make_sdesc_sw128(sbase + kOffW + wslot * kWStage, 16, 1024);
          const uint32_t d_tmem = tmem_base + nh * p.bnc;
#pragma unroll
          for (int k = 0; k < kKC / 16; ++k) ptx::umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          ptx::tc_commit_a(w_empty + 8 * wslot);
          if (++wslot == kWStages) {
            wslot = 0;
            wphase ^= 1;
          }
        }
        ptx::tc_commit_a(a_empty + 8 * s);
      }
      ptx::tc_commit_a(acc_full);
    }
  } else {
    // ------------------------------------------------------------------ depth-wise producers
    const int pw = warp - kCtrlWarps;
    const int strip = pw & (kStripWarps - 1);
    const int group = pw / kStripWarps;
    const uint32_t a_lane = ((lane & 3) << 2);
    const uint32_t chunk = static_cast<uint32_t>(lane >> 2);
#pragma unroll 1
    for (int kb = group; kb < p.num_kb; kb += kGroups) {
      const int s = kb & 1;  // A slot (= group)
      const uint32_t ph = (kb >> 1) & 1;
      const int gs = kb % kGStages;
      ptx::mbar_wait_a(g_full + 8 * gs, (kb / kGStages) & 1);
      const uint32_t tp = sbase + kOffT + gs * kTapBytes + lane * 8;
      float2 w[kTaps];
#pragma unroll
      for (int k = 0; k < kTaps; ++k) w[k] = lds64f(tp + k * (kKC * 4));
      const float2 bias = lds64f(tp + kTaps * (kKC * 4));
      float2 acc[kStrip];
#pragma unroll
      for (int o = 0; o < kStrip; ++o) acc[o] = bias;
      const uint32_t gp = sbase + kOffG + gs * kGStage + (strip * kStrip) * 128 + lane * 4;
#pragma unroll
      for (int j = 0; j < kStrip + kTaps - 1; ++j) {
        const uint32_t u = lds32u(gp + j * 128);
        const float2 vv = make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
#pragma unroll
        for (int o = 0; o < kStrip; ++o) {
          const int k = j - o;
          if (k >= 0 && k < kTaps) acc[o] = ffma2(w[k], vv, acc[o]);
        }
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_a(g_empty + 8 * gs);  // halo tile and taps of this stage are in registers
      ptx::mbar_wait_a(a_empty + 8 * s, ph ^ 1);           // the MMAs that read this A slot two k-blocks ago are done
      const uint32_t ap = sbase + kOffA + s * kAStage + (strip * kStrip) * 128 + a_lane;
#pragma unroll
      for (int o = 0; o < kStrip; ++o) {
        const uint32_t v = ptx::pack_bf16x2(swish_fast(acc[o].x), swish_fast(acc[o].y));
        sts32u(ap + o * 128 + ((chunk ^ static_cast<uint32_t>(o & 7)) << 4), v);
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_a(a_full + 8 * s);
    }

    // ------------------------------------------------------------------ epilogue: x += acc + b2
    const int quarter = warp & 3;           // TMEM lanes this warp may read
    const int colgroup = pw >> 2;            // 0..3: takes boxes colgroup, colgroup + 4, ... (its 4 warps = 4 quarters)
    const int row0 = t0 + quarter * 32;
    ptx::mbar_wait_a(acc_full, 0);
    ptx::tc_fence_after();
    if (row0 < p.T) {
      uint8_t* stage_base = smem + pw * 8192;
      const uint32_t swz = static_cast<uint32_t>(lane & 7);
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
      const uint32_t stage_a = ptx::smem_u32(stage_base), bias_a = ptx::smem_u32(smem + kOffBias);
      uint32_t cnt = 0;
      const int boxes = p.d / 32;
#pragma unroll 1
      for (int box = colgroup; box < boxes; box += kProdWarps / 4, ++cnt) {
        uint8_t* sbuf = stage_base + (cnt & 1u) * 4096;
        uint32_t v[32];
        ptx::tmem_ld_x32(t_addr + box * 32, v);
        if (lane == 0) ptx::bulk_wait_read<1>();  // the reduce that last read this staging box has drained it
        __syncwarp();
        ptx::tc_wait_ld();
        // shared-space accesses by 32-bit address (through the rounded-up generic pointer these were LD.E / ST.E)
        const uint32_t srow = stage_a + (cnt & 1u) * 4096 + lane * 128;
        const uint32_t bs = bias_a + 4 * box * 32;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 bb = ptx::lds_f32x4(bs + 16 * j);
          ptx::sts128(srow + ((static_cast<uint32_t>(j) ^ swz) << 4), __float_as_uint(__uint_as_float(v[4 * j]) + bb.x),
                      __float_as_uint(__uint_as_float(v[4 * j + 1]) + bb.y), __float_as_uint(__uint_as_float(v[4 * j + 2]) + bb.z),
                      __float_as_uint(__uint_as_float(v[4 * j + 3]) + bb.w));
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          ptx::tma_reduce_add_3d(&tmO, sbuf, box * 32, row0, b);
          ptx::bulk_commit();
        }
      }
      // the staging boxes must outlive their reads; the global side of the reductions completes with the grid
      if (lane == 0) ptx::bulk_wait_read<0>();
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

}  // namespace

bool dw_pw_supported(int d) { return d >= 64 && d % 64 == 0 && d <= 512; }

int launch_dw_pw(const DwPwDesc& c, cudaStream_t st, std::string* err) {
  if (c.B <= 0 || c.T <= 0) return 0;
  if (!dw_pw_supported(c.d)) {
    if (err) *err = "dw_pw: d_model must be a multiple of 64 and <= 512";
    return -1;
  }
  const int d = c.d;
  DwPwParams p{};
  p.T = c.T;
  p.d = d;
  p.num_kb = d / kKC;
  p.nc = d > 256 ? 2 : 1;
  p.bnc = d / p.nc;  // 32 * (d / 64) or d: a multiple of 16, <= 256
  p.tblocks = (c.T + kTileT - 1) / kTileT;
  p.tmem_cols = 32;
  while (p.tmem_cols < static_cast<uint32_t>(d)) p.tmem_cols <<= 1;
  p.bias2 = c.bias2;
  CUtensorMap tmG, tmT, tmW, tmO;
  {
    uint64_t dims[3] = {static_cast<uint64_t>(d), static_cast<uint64_t>(c.T), static_cast<uint64_t>(c.B)};
    uint64_t strides[2] = {static_cast<uint64_t>(d) * 2, static_cast<uint64_t>(d) * 2 * c.T};
    uint32_t box[3] = {kKC, kGRows, 1};
    if (!encode_tmap_ex(&tmG, c.g, false, 3, dims, strides, box, false, err)) return -1;
  }
  {
    uint64_t dims[2] = {static_cast<uint64_t>(d), 32};
    uint64_t strides[1] = {static_cast<uint64_t>(d) * 4};
    uint32_t box[2] = {kKC, 32};
    if (!encode_tmap_ex(&tmT, c.taps32, true, 2, dims, strides, box, false, err)) return -1;
  }
  {
    uint64_t dims[2] = {static_cast<uint64_t>(d), static_cast<uint64_t>(d)};
    uint64_t strides[1] = {static_cast<uint64_t>(d) * 2};
    uint32_t box[2] = {kKC, static_cast<uint32_t>(p.bnc)};
    if (!encode_tmap_bf16(&tmW, c.W, 2, dims, strides, box, err)) return -1;
  }
  {
    uint64_t dims[3] = {static_cast<uint64_t>(d), static_cast<uint64_t>(c.T), static_cast<uint64_t>(c.B)};
    uint64_t strides[2] = {static_cast<uint64_t>(d) * 4, static_cast<uint64_t>(d) * 4 * c.T};
    uint32_t box[3] = {32, 32, 1};
    if (!encode_tmap(&tmO, c.x, true, 3, dims, strides, box, err)) return -1;
  }
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63]) {
    const cudaError_t e = cudaFuncSetAttribute(dw_pw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTotal);
    if (e != cudaSuccess) {
      if (err) *err = std::string("cudaFuncSetAttribute(dw_pw): ") + cudaGetErrorString(e);
      return static_cast<int>(e);
    }
    configured[dev & 63] = true;
  }
  const cudaError_t e =
      launch_pdl(dw_pw_kernel, dim3(c.B * p.tblocks), dim3(kThreads), kSmemTotal, st, tmG, tmT, tmW, tmO, p);
  if (e != cudaSuccess) {
    if (err) *err = std::string("dw_pw launch: ") + cudaGetErrorString(e);
    return static_cast<int>(e);
  }
  return 0;
}

}  // namespace cfb
