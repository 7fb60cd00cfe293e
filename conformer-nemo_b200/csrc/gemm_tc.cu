// tcgen05 GEMM for sm_100a:  D (M x N) = A (M x K, bf16) * W^T (W: N x K, bf16), fp32 accumulation in TMEM,
// fused epilogue (epilogue.cuh).  Also the implicit-GEMM form of the strided 3x3 subsampling convolution.
//
// One persistent CTA per SM, 320 threads, warp-specialised:
//   warp 0      TMA producer (one lane): A and W tiles, 128-byte swizzle, STAGES-deep mbarrier ring
//   warp 1      MMA issuer (one lane): tcgen05.mma cta_group::1, 128 x BN x 16 per instruction, BLOCK_K = 64
//   warps 2..9  epilogue (two warps per TMEM lane quarter, alternating output boxes): tcgen05.ld 32x32b (thread = output row), bias / activation / mask in registers, values
//               staged into a 128-byte-swizzled smem box per warp (32 rows x 128 B, double-buffered) and written
//               with TMA stores -- plain stores for bf16 / fp32 outputs, cp.reduce.async.bulk (.add.f32) into the
//               fp32 residual stream -- so every global write is a full 128-byte line
// Operand bytes in flight decide the sustained rate (TMA latency ~1 us vs 270 ns per 48 KB k-block at full tensor
// rate): 256-wide tiles run 4 stages (192 KB in flight) and pay for the fourth with single-buffered output staging.
// The accumulator is double-buffered in TMEM (2 x BN columns) so the epilogue of tile i overlaps the main loop
// of tile i+1.  M/N/K tails are handled by TMA zero fill on the load side and TMA clipping on the store side.
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"
#include "epilogue.cuh"
#include "ptx.cuh"

namespace cfb {

namespace {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;  // 64 bf16 = one 128-byte swizzle row
constexpr int kEpiWarps = 8;  // two per TMEM lane quarter
constexpr int kThreads = 64 + 32 * kEpiWarps;

struct TcParams {
  int num_tiles;
  int num_n_tiles;
  int num_k_blocks;
  // implicit-GEMM convolution (CONV = true)
  int conv_cchunks;   // k-blocks per filter tap = ceil(C_in / 64)
  int conv_cin;
  int conv_tblocks;   // output tiles per sequence along time (32 frames each)
  int conv_fblocks;   // output tiles along frequency (4 bins each)
  int conv_To, conv_Fo;
  EpiParams ep;
};

// SBUF = staging boxes per epilogue warp (2 = double-buffered TMA stores; 1 frees 32 KB for one more operand stage)
template <int BN, int STAGES, int SBUF = ((BN == 256 && STAGES >= 4) ? 1 : 2)>
struct SmemLayout {
  static constexpr int kSBuf = SBUF;
  static constexpr int kABytes = kBlockM * kBlockK * 2;
  static constexpr int kBBytes = BN * kBlockK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStagingOffset = STAGES * kStageBytes;  // per epilogue warp: 2 buffers x (32 rows x 128 B)
  static constexpr int kStagingBytes = kEpiWarps * SBUF * 4096;
  static constexpr int kBarOffset = kStagingOffset + kStagingBytes;
  static constexpr int kBiasOffset = kBarOffset + 256;          // float [2][BN]: the current / next tile's bias
  static constexpr int kNeeded = kBiasOffset + 2 * BN * 4;
  // operand tiles need 1024-byte alignment; ask for the slack when it fits (the kernel traps if it did not get it)
  static constexpr int kTotal = kNeeded + 1024 <= 227 * 1024 ? kNeeded + 1024 : 227 * 1024;
};

template <int BN, int STAGES, int EPI, typename TOut, bool CONV>
__global__ void __launch_bounds__(kThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmO, const TcParams p) {
  using L = SmemLayout<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  if (static_cast<int>(smem - smem_raw) + L::kNeeded > L::kTotal) __trap();  // alignment slack did not fit
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* acc_full = empty_bar + STAGES;  // [2]
  uint64_t* acc_empty = acc_full + 2;       // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t kTmemCols = 2 * BN;  // 128 / 256 / 512: a power of two >= 32

  if (warp == 0) {
    if (lane == 0) {
      ptx::prefetch_tmap(&tmA);
      ptx::prefetch_tmap(&tmB);
      ptx::prefetch_tmap(&tmO);
      for (int s = 0; s < STAGES; ++s) {
        ptx::mbar_init(&full_bar[s], 1);
        ptx::mbar_init(&empty_bar[s], 1);
      }
      for (int b = 0; b < 2; ++b) {
        ptx::mbar_init(&acc_full[b], 1);
        ptx::mbar_init(&acc_empty[b], 32 * kEpiWarps);
      }
      ptx::fence_mbar_init();
    }
    __syncwarp();
    ptx::tmem_alloc(tmem_slot, kTmemCols);
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();  // the next kernel may begin its own setup
  pdl_wait();               // the previous kernel's output (A, the residual stream) is complete from here on

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const int n_blk = tile % p.num_n_tiles;
        const int m_blk = tile / p.num_n_tiles;
        for (int kb = 0; kb < p.num_k_blocks; ++kb) {
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
          ptx::mbar_arrive_expect_tx(&full_bar[stage], L::kStageBytes);
          uint8_t* sa = smem + stage * L::kStageBytes;
          uint8_t* sb = sa + L::kABytes;
          if constexpr (CONV) {
            const int fb = m_blk % p.conv_fblocks;
            const int tb = (m_blk / p.conv_fblocks) % p.conv_tblocks;
            const int b = m_blk / (p.conv_fblocks * p.conv_tblocks);
            const int tap = kb / p.conv_cchunks;
            const int cc = kb - tap * p.conv_cchunks;
            const int kh = tap / 3, kw = tap - kh * 3;
            // input index 2*o + k - 1: k = 1 -> even plane, same index; k = 0 -> odd plane, index o-1; k = 2 -> odd, o
            const int plane = ((kh == 1) ? 0 : 2) + ((kw == 1) ? 0 : 1);
            const int tcoord = tb * 32 - (kh == 0 ? 1 : 0);
            const int fcoord = fb * 4 - (kw == 0 ? 1 : 0);
            ptx::tma_load_5d(sa, &tmA, &full_bar[stage], cc * 64, fcoord, tcoord, plane, b);
            ptx::tma_load_2d(sb, &tmB, &full_bar[stage], tap * p.conv_cin + cc * 64, n_blk * BN);
          } else {
            ptx::tma_load_2d(sa, &tmA, &full_bar[stage], kb * kBlockK, m_blk * kBlockM);
            ptx::tma_load_2d(sb, &tmB, &full_bar[stage], kb * kBlockK, n_blk * BN);
          }
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16(kBlockM, BN, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1;
        ptx::mbar_wait(&acc_empty[buf], ((it >> 1) & 1) ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * BN;
        for (int kb = 0; kb < p.num_k_blocks; ++kb) {
          ptx::mbar_wait(&full_bar[stage], phase);
          ptx::tc_fence_after();
          const uint32_t sa = ptx::smem_u32(smem + stage * L::kStageBytes);
          const uint64_t da = ptx::make_sdesc_sw128(sa, 16, 1024);
          const uint64_t db = ptx::make_sdesc_sw128(sa + L::kABytes, 16, 1024);
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) {
            // +32 bytes per K step inside the 128-byte swizzle row (descriptor address field is in 16-byte units)
            ptx::umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          ptx::tc_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs have read it
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        ptx::tc_commit(&acc_full[buf]);
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps
    constexpr bool kFast = OutTraits<TOut>::kFast;
    constexpr int kBoxCols = 128 / static_cast<int>(sizeof(TOut));           // output columns per 128-byte box row
    constexpr int kAccPerBox = (EPI == EPI_GLU) ? 2 * kBoxCols : kBoxCols;   // accumulator columns feeding one box
    constexpr int kChunks = kAccPerBox / 32;
    constexpr int kBoxes = BN / kAccPerBox;
    static_assert(kBoxes >= 1, "tile narrower than one output box");
    const int quarter = warp & 3;        // TMEM lanes this warp may read: [32*quarter, +32)
    const int half = (warp - 2) >> 2;    // which of the quarter's two warps: takes boxes half, half+2, ...
    const int row_in_tile = quarter * 32 + lane;
    uint8_t* stage_base = smem + L::kStagingOffset + (warp - 2) * (L::kSBuf * 4096);
    // 32-bit shared-window addresses for the staging rows and the bias: through the rounded-up generic pointer the compiler
    // cannot prove the address space and emits generic LD.E / ST.E (long-scoreboard) for every access of the epilogue
    const uint32_t stage_a = ptx::smem_u32(stage_base), bias_a0 = ptx::smem_u32(smem + L::kBiasOffset);
    const uint32_t swz = static_cast<uint32_t>(lane & 7);
    uint32_t box_counter = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      const int n_blk = tile % p.num_n_tiles;
      const int m_blk = tile / p.num_n_tiles;
      long long out_row;
      bool row_ok;
      int cv_f0 = 0, cv_t0 = 0, cv_b = 0;
      if constexpr (CONV) {
        const int fb = m_blk % p.conv_fblocks;
        const int tb = (m_blk / p.conv_fblocks) % p.conv_tblocks;
        cv_b = m_blk / (p.conv_fblocks * p.conv_tblocks);
        const int t = tb * 32 + (row_in_tile >> 2);
        const int f = fb * 4 + (row_in_tile & 3);
        cv_f0 = fb * 4;
        cv_t0 = tb * 32 + quarter * 8;
        row_ok = (t < p.conv_To) && (f < p.conv_Fo);
        out_row = (static_cast<long long>(cv_b) * p.conv_To + t) * p.conv_Fo + f;
      } else {
        out_row = static_cast<long long>(m_blk) * kBlockM + row_in_tile;
        row_ok = out_row < p.ep.M;
      }
      const bool keep = row_ok ? epi_keep<EPI>(p.ep, out_row) : true;  // its load is in flight during the accumulator wait
      // stage this tile's bias (BN floats) in shared memory while the accumulator is still being computed
      const uint32_t bias_a = bias_a0 + buf * BN * 4;
      {
        const int e = static_cast<int>(threadIdx.x) - 64;
        if (e < BN) {
          const int col = n_blk * BN + e;
          ptx::sts_f32(bias_a + 4 * e, (p.ep.bias != nullptr && col < p.ep.N) ? __ldg(p.ep.bias + col) : 0.f);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
      }
      ptx::mbar_wait(&acc_full[buf], (it >> 1) & 1);
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + buf * BN;
#pragma unroll 1
      for (int box = half; box < kBoxes; box += kEpiWarps / 4) {
        const int acc_col0 = n_blk * BN + box * kAccPerBox;
        if (acc_col0 >= p.ep.N) break;  // warp-uniform: nothing of this box is inside the matrix
        const int n_pass = (EPI == EPI_QKV && acc_col0 < p.ep.qkv_dp) ? 2 : 1;
#pragma unroll 1
        for (int pass = 0; pass < n_pass; ++pass) {
          uint8_t* sbuf = stage_base + (L::kSBuf == 2 ? (box_counter & 1u) * 4096 : 0u);
          if (lane == 0) {  // the store that last read this buffer has drained it
            if constexpr (L::kSBuf == 2) ptx::bulk_wait_read<1>();
            else ptx::bulk_wait_read<0>();
          }
          __syncwarp();
          const uint32_t srow = stage_a + static_cast<uint32_t>(sbuf - stage_base) + lane * 128;
#pragma unroll
          for (int ch = 0; ch < kChunks; ++ch) {
            uint32_t v[32];
            ptx::tmem_ld_x32(t_addr + box * kAccPerBox + ch * 32, v);
            ptx::tc_wait_ld();
            float acc[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[j] = __uint_as_float(v[j]);
            if (row_ok) {
              if (EPI == EPI_QKV && pass == 1) {
                epi_compute<EPI, kFast>(p.ep, out_row, acc_col0 + ch * 32, acc, pass);  // q + v: bias2 from global
              } else {
                float b[32];
                const uint32_t bs = bias_a + 4 * (box * kAccPerBox + ch * 32);
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float4 t = ptx::lds_f32x4(bs + 16 * j);
                  b[4 * j] = t.x, b[4 * j + 1] = t.y, b[4 * j + 2] = t.z, b[4 * j + 3] = t.w;
                }
                epi_math_keep<EPI, kFast>(p.ep, keep, acc, b);
              }
            }
            if constexpr (sizeof(TOut) == 4) {
#pragma unroll
              for (int j = 0; j < 8; ++j)
                ptx::sts128(srow + ((static_cast<uint32_t>(j) ^ swz) << 4), __float_as_uint(acc[4 * j]), __float_as_uint(acc[4 * j + 1]),
                            __float_as_uint(acc[4 * j + 2]), __float_as_uint(acc[4 * j + 3]));
            } else {
              constexpr int kPieces = (EPI == EPI_GLU) ? 2 : 4;  // 16-byte pieces produced by this chunk
#pragma unroll
              for (int j = 0; j < kPieces; ++j) {
                uint4 u;
                u.x = ptx::pack_bf16x2(acc[8 * j + 0], acc[8 * j + 1]);
                u.y = ptx::pack_bf16x2(acc[8 * j + 2], acc[8 * j + 3]);
                u.z = ptx::pack_bf16x2(acc[8 * j + 4], acc[8 * j + 5]);
                u.w = ptx::pack_bf16x2(acc[8 * j + 6], acc[8 * j + 7]);
                ptx::sts128(srow + ((static_cast<uint32_t>(ch * kPieces + j) ^ swz) << 4), u.x, u.y, u.z, u.w);
              }
            }
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if constexpr (CONV) {
              ptx::tma_store_4d(&tmO, sbuf, acc_col0, cv_f0, cv_t0, cv_b);
            } else {
              const int row0 = m_blk * kBlockM + quarter * 32;
              if constexpr (EPI == EPI_RESID) {
                ptx::tma_reduce_add_2d(&tmO, sbuf, acc_col0, row0);
              } else if constexpr (EPI == EPI_QKV) {
                const int oc = (pass == 1 || acc_col0 >= p.ep.qkv_dp) ? acc_col0 + p.ep.qkv_dp : acc_col0;
                ptx::tma_store_2d(&tmO, sbuf, oc, row0);
              } else if constexpr (EPI == EPI_GLU) {
                ptx::tma_store_2d(&tmO, sbuf, acc_col0 >> 1, row0);
              } else {
                ptx::tma_store_2d(&tmO, sbuf, acc_col0, row0);
              }
            }
            ptx::bulk_commit();
          }
          ++box_counter;
        }
      }
      ptx::tc_fence_before();
      ptx::mbar_arrive(&acc_empty[buf]);
    }
    if (lane == 0) ptx::bulk_wait_read<0>();  // staging boxes outlive their reads; the global side completes with the grid
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

int g_num_sms = 0;
int num_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}

template <int BN, int STAGES, int EPI, typename TOut, bool CONV>
int launch_instance(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO, const TcParams& p,
                    cudaStream_t st, std::string* err) {
  using L = SmemLayout<BN, STAGES>;
  auto kern = gemm_tc_kernel<BN, STAGES, EPI, TOut, CONV>;
  static bool configured[64] = {};  // per instantiation and device
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal);
    if (e != cudaSuccess) {
      if (err) *err = std::string("cudaFuncSetAttribute(gemm_tc): ") + cudaGetErrorString(e);
      return static_cast<int>(e);
    }
    configured[dev & 63] = true;
  }
  const int grid = p.num_tiles < num_sms() ? p.num_tiles : num_sms();
  cudaError_t e = launch_pdl(kern, dim3(grid), dim3(kThreads), L::kTotal, st, tmA, tmB, tmO, p);
  if (e != cudaSuccess) {
    if (err) *err = std::string("gemm_tc launch: ") + cudaGetErrorString(e);
    return static_cast<int>(e);
  }
  return 0;
}

template <int BN, int STAGES, bool CONV>
int dispatch_epi(int epi, bool out_bf16, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO,
                 const TcParams& p, cudaStream_t st, std::string* err) {
  if constexpr (CONV) {
    return launch_instance<BN, STAGES, EPI_RELU, bf16, true>(tmA, tmB, tmO, p, st, err);
  } else {
    switch (epi) {
      case EPI_LINEAR:
        return out_bf16 ? launch_instance<BN, STAGES, EPI_LINEAR, bf16, false>(tmA, tmB, tmO, p, st, err)
                        : launch_instance<BN, STAGES, EPI_LINEAR, float, false>(tmA, tmB, tmO, p, st, err);
      case EPI_SWISH:
        return launch_instance<BN, STAGES, EPI_SWISH, bf16, false>(tmA, tmB, tmO, p, st, err);
      case EPI_RELU:
        return launch_instance<BN, STAGES, EPI_RELU, bf16, false>(tmA, tmB, tmO, p, st, err);
      case EPI_RESID:
        return launch_instance<BN, STAGES, EPI_RESID, float, false>(tmA, tmB, tmO, p, st, err);
      case EPI_QKV:
        return launch_instance<BN, STAGES, EPI_QKV, bf16, false>(tmA, tmB, tmO, p, st, err);
      case EPI_GLU:
        return launch_instance<BN, STAGES, EPI_GLU, bf16, false>(tmA, tmB, tmO, p, st, err);
      default:
        if (err) *err = "gemm_tc: unknown epilogue";
        return -1;
    }
  }
}

}  // namespace

int launch_gemm_tc(const GemmDesc& g, cudaStream_t st, std::string* err) {
  if (g.M <= 0 || g.N <= 0 || g.K <= 0) return 0;
  if ((g.lda % 8) || (g.ldw % 8) || (g.K % 8)) {
    if (err) *err = "gemm_tc: K and leading dimensions must be multiples of 8 (16-byte TMA strides)";
    return -1;
  }
  const int m_tiles = (g.M + kBlockM - 1) / kBlockM;
  // Small M (a rank's share of a sharded batch, one of its groups): when 128-wide tiles still fit in one wave, every CTA
  // owns ONE tile and its time is fill + K loop + epilogue in series -- 128-wide tiles double the CTAs and halve both the
  // operand bytes per k-block and the epilogue per CTA (the tiles are latency-bound there, not operand-bound).  This
  // also takes precedence over the CTA-pair kernel, whose 256 x 256 tiles are the coarsest.
  const bool small_m = g.N % 256 == 0 && 2 * m_tiles * (g.N / 256) <= num_sms();
  if (!small_m) {
    // CTA pairs (gemm_tc2.cu): CFB_GEMM_2CTA=0 never, =1 whenever the shape allows, unset = the measured default
    const char* v2 = getenv("CFB_GEMM_2CTA");
    const int mode = v2 ? atoi(v2) : -1;
    // measured (r02j/l, M = 16000): N 2048 K 512 plain 35.0 -> 31.6 us, qkv 33.1 -> 29.6, linear1+swish 36.2 -> 35.7
    // (its MUFU-bound epilogue takes over), pw1+glu 21.3 -> 22.1, K = 2048 neutral
    if (mode != 0 && gemm_tc2_supported(g) && (mode == 1 || (g.K <= 1024 && g.N >= 1536))) return launch_gemm_tc2(g, st, err);
  }
  // tile width: 256 for wide outputs (256-wide tiles halve the re-reads of A: the kernel is bound by L2->SM bandwidth,
  // not by the tensor pipe), else 128
  int bn = 128;
  if (g.N % 256 == 0 && !small_m) bn = 256;
  const int n_tiles = (g.N + bn - 1) / bn;

  CUtensorMap tmA, tmB;
  {
    uint64_t dims[2] = {static_cast<uint64_t>(g.K), static_cast<uint64_t>(g.M)};
    uint64_t strides[1] = {static_cast<uint64_t>(g.lda) * 2};
    uint32_t box[2] = {kBlockK, kBlockM};
    if (!encode_tmap_bf16(&tmA, g.A, 2, dims, strides, box, err)) return -1;
  }
  {
    uint64_t dims[2] = {static_cast<uint64_t>(g.K), static_cast<uint64_t>(g.N)};
    uint64_t strides[1] = {static_cast<uint64_t>(g.ldw) * 2};
    uint32_t box[2] = {kBlockK, static_cast<uint32_t>(bn)};
    if (!encode_tmap_bf16(&tmB, g.W, 2, dims, strides, box, err)) return -1;
  }
  TcParams p{};
  p.num_n_tiles = n_tiles;
  p.num_tiles = m_tiles * n_tiles;
  p.num_k_blocks = (g.K + kBlockK - 1) / kBlockK;
  p.ep = g.ep;
  p.ep.M = g.M;
  p.ep.N = g.N;
  // output map: 32-row boxes, 128 bytes wide (one epilogue warp's slab)
  CUtensorMap tmO;
  {
    const bool f32 = !g.out_bf16 || g.epi == EPI_RESID;
    uint64_t cols = static_cast<uint64_t>(g.N);
    if (g.epi == EPI_QKV) cols = static_cast<uint64_t>(g.N) + g.ep.qkv_dp;  // [q+u | q+v | k | v]
    if (g.epi == EPI_GLU) cols = static_cast<uint64_t>(g.N) / 2;
    if ((g.ep.ldo * (f32 ? 4 : 2)) % 16) {
      if (err) *err = "gemm_tc: output leading dimension must be a multiple of 16 bytes";
      return -1;
    }
    uint64_t dims[2] = {cols, static_cast<uint64_t>(g.M)};
    uint64_t strides[1] = {static_cast<uint64_t>(g.ep.ldo) * (f32 ? 4 : 2)};
    uint32_t box[2] = {f32 ? 32u : 64u, 32u};
    if (!encode_tmap(&tmO, g.ep.out, f32, 2, dims, strides, box, err)) return -1;
  }
  // long K: the mainloop dominates -> 4 operand stages, single-buffered staging; short K: a tile's epilogue takes as
  // long as its mainloop and a TMA store holds its staging box ~1500 cycles -> 3 stages, double-buffered staging
  if (bn == 256 && p.num_k_blocks >= 16) return dispatch_epi<256, 4, false>(g.epi, g.out_bf16, tmA, tmB, tmO, p, st, err);
  if (bn == 256) return dispatch_epi<256, 3, false>(g.epi, g.out_bf16, tmA, tmB, tmO, p, st, err);
  return dispatch_epi<128, 5, false>(g.epi, g.out_bf16, tmA, tmB, tmO, p, st, err);
}

int launch_conv_tc(const ConvDesc& c, cudaStream_t st, std::string* err) {
  if (c.C_in % 8 || c.C_out % 8) {
    if (err) *err = "conv_tc: channel counts must be multiples of 8";
    return -1;
  }
  CUtensorMap tmA, tmB;
  {
    // [B][plane 4][Th][Fh][C] -> dims innermost first
    uint64_t dims[5] = {static_cast<uint64_t>(c.C_in), static_cast<uint64_t>(c.Fh), static_cast<uint64_t>(c.Th), 4,
                        static_cast<uint64_t>(c.B)};
    uint64_t s1 = static_cast<uint64_t>(c.C_in) * 2;
    uint64_t strides[4] = {s1, s1 * c.Fh, s1 * c.Fh * c.Th, s1 * c.Fh * c.Th * 4};
    uint32_t box[5] = {64, 4, 32, 1, 1};
    if (!encode_tmap_bf16(&tmA, c.y_in, 5, dims, strides, box, err)) return -1;
  }
  const int K = 9 * c.C_in;
  const int bn = (c.C_out % 256 == 0) ? 256 : 128;
  {
    uint64_t dims[2] = {static_cast<uint64_t>(K), static_cast<uint64_t>(c.C_out)};
    uint64_t strides[1] = {static_cast<uint64_t>(K) * 2};
    uint32_t box[2] = {kBlockK, static_cast<uint32_t>(bn)};
    if (!encode_tmap_bf16(&tmB, c.W, 2, dims, strides, box, err)) return -1;
  }
  TcParams p{};
  p.conv_cin = c.C_in;
  p.conv_cchunks = (c.C_in + 63) / 64;
  p.conv_tblocks = (c.To + 31) / 32;
  p.conv_fblocks = (c.Fo + 3) / 4;
  p.conv_To = c.To;
  p.conv_Fo = c.Fo;
  p.num_n_tiles = (c.C_out + bn - 1) / bn;
  p.num_tiles = c.B * p.conv_tblocks * p.conv_fblocks * p.num_n_tiles;
  p.num_k_blocks = 9 * p.conv_cchunks;
  p.ep.bias = c.bias;
  p.ep.out = c.y_out;
  p.ep.ldo = c.C_out;
  p.ep.M = c.B * c.To * c.Fo;
  p.ep.N = c.C_out;
  CUtensorMap tmO;
  {
    // y2 [B][To][Fo][C]: a warp's 32 accumulator rows are 8 frames x 4 bins -> one 4-D box
    uint64_t dims[4] = {static_cast<uint64_t>(c.C_out), static_cast<uint64_t>(c.Fo), static_cast<uint64_t>(c.To),
                        static_cast<uint64_t>(c.B)};
    uint64_t s1 = static_cast<uint64_t>(c.C_out) * 2;
    uint64_t strides[3] = {s1, s1 * c.Fo, s1 * c.Fo * c.To};
    uint32_t box[4] = {64, 4, 8, 1};
    if (!encode_tmap_bf16(&tmO, c.y_out, 4, dims, strides, box, err)) return -1;
  }
  if (bn == 256) return dispatch_epi<256, 4, true>(EPI_RELU, true, tmA, tmB, tmO, p, st, err);
  return dispatch_epi<128, 5, true>(EPI_RELU, true, tmA, tmB, tmO, p, st, err);
}

}  // namespace cfb
