// tcgen05 GEMM on CTA PAIRS (cta_group::2):  D (M x N) = A (M x K, bf16) * W^T (W: N x K, bf16), fp32 accumulation in
// TMEM, the fused epilogues of epilogue.cuh.  Same warp roles as gemm_tc.cu, but two CTAs on the two SMs of a TPC own
// one 256 x 256 tile: each CTA loads ITS 128 rows of A and ITS 128 rows of the 256-row W box (32 KB per k-block
// instead of 48 KB for the same 128 x 256 x 64 MACs per SM), the leader CTA issues 256 x 256 x 16 MMAs that read both
// halves, and each CTA's epilogue drains its own 128 accumulator rows.
// Why: gemm_tc's K = 512 / 2048 GEMMs are bound by operand bytes in flight (shared memory holds 3-4 stages of 48 KB
// against ~1 us of L2 latency); a pair keeps 5 stages of 32 KB in flight = 5 k-blocks of tensor work instead of 3.
//   warp 0      TMA producer (both CTAs; transaction bytes are counted on the leader's full barrier)
//   warp 1      MMA issuer (leader CTA only); tcgen05.commit multicasts "slot free" / "accumulator full" to both CTAs
//   warps 2..9  epilogue (both CTAs, own rows); "accumulator drained" arrives on the leader's barrier from both
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"
#include "epilogue.cuh"
#include "ptx.cuh"

namespace cfb {

namespace {

constexpr int kBlockM = 128;   // rows per CTA (256 per pair)
constexpr int kBlockK = 64;
constexpr int kBN = 256;       // tile width (128 W rows per CTA)
constexpr int kEpiWarps = 8;
constexpr int kThreads = 64 + 32 * kEpiWarps;
constexpr int kStages = 5;
constexpr int kABytes = kBlockM * kBlockK * 2;
constexpr int kBBytes = (kBN / 2) * kBlockK * 2;
constexpr int kStageBytes = kABytes + kBBytes;         // 32 KB
constexpr int kStagingOffset = kStages * kStageBytes;  // per epilogue warp: 2 x (32 rows x 128 B)
constexpr int kStagingBytes = kEpiWarps * 2 * 4096;
constexpr int kBarOffset = kStagingOffset + kStagingBytes;
constexpr int kBiasOffset = kBarOffset + 256;          // float [2][kBN]
constexpr int kNeeded = kBiasOffset + 2 * kBN * 4;
constexpr int kTotal = kNeeded + 1024 <= 227 * 1024 ? kNeeded + 1024 : 227 * 1024;
static_assert(kNeeded <= 227 * 1024, "shared memory budget");

struct Tc2Params {
  int num_tiles;      // 256 x 256 tiles
  int num_n_tiles;
  int num_k_blocks;
  EpiParams ep;
};

template <int EPI, typename TOut>
__global__ void __launch_bounds__(kThreads, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmO, const Tc2Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  if (static_cast<int>(smem - smem_raw) + kNeeded > kTotal) __trap();  // alignment slack did not fit
  const uint32_t sbase = ptx::smem_u32(smem);
  const uint32_t full_bar = sbase + kBarOffset;          // [kStages] leader: 64 KB of both CTAs' loads landed
  const uint32_t empty_bar = full_bar + 8 * kStages;     // [kStages] both CTAs: the MMAs that read the slot are done
  const uint32_t acc_full = empty_bar + 8 * kStages;     // [2] both CTAs
  const uint32_t acc_empty = acc_full + 16;              // [2] leader: 16 warp arrivals (8 per CTA)
  const uint32_t tmem_slot = acc_empty + 16;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const int pair = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;
  constexpr uint32_t kTmemCols = 2 * kBN;

  if (warp == 0) {
    if (lane == 0) {
      ptx::prefetch_tmap(&tmA);
      ptx::prefetch_tmap(&tmB);
      ptx::prefetch_tmap(&tmO);
      for (int s = 0; s < kStages; ++s) {
        ptx::mbar_init_a(full_bar + 8 * s, 1);
        ptx::mbar_init_a(empty_bar + 8 * s, 1);
      }
      for (int b = 0; b < 2; ++b) {
        ptx::mbar_init_a(acc_full + 8 * b, 1);
        ptx::mbar_init_a(acc_empty + 8 * b, 2 * kEpiWarps);
      }
      ptx::fence_mbar_init();
    }
    __syncwarp();
    ptx::tmem_alloc_2cta(tmem_slot, kTmemCols);
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();  // both CTAs' barriers are initialised before anybody signals across the pair
  ptx::tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");
  pdl_launch_dependents();
  pdl_wait();

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (both CTAs)
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = pair; tile < p.num_tiles; tile += num_pairs) {
        const int n_blk = tile % p.num_n_tiles;
        const int m_blk = tile / p.num_n_tiles;
        const int row_a = (2 * m_blk + static_cast<int>(rank)) * kBlockM;
        const int row_b = n_blk * kBN + static_cast<int>(rank) * (kBN / 2);
        for (int kb = 0; kb < p.num_k_blocks; ++kb) {
          ptx::mbar_wait_a(empty_bar + 8 * stage, phase ^ 1);
          if (rank == 0) ptx::mbar_arrive_expect_tx_a(full_bar + 8 * stage, 2 * kStageBytes);
          const uint32_t sa = sbase + stage * kStageBytes;
          ptx::tma_load_2d_2cta(sa, &tmA, full_bar + 8 * stage, kb * kBlockK, row_a);
          ptx::tma_load_2d_2cta(sa + kABytes, &tmB, full_bar + 8 * stage, kb * kBlockK, row_b);
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only)
    if (rank == 0 && lane == 0) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16(2 * kBlockM, kBN, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = pair; tile < p.num_tiles; tile += num_pairs, ++it) {
        const int buf = it & 1;
        ptx::mbar_wait_a(acc_empty + 8 * buf, ((it >> 1) & 1) ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * kBN;
        for (int kb = 0; kb < p.num_k_blocks; ++kb) {
          ptx::mbar_wait_a(full_bar + 8 * stage, phase);
          ptx::tc_fence_after();
          const uint32_t sa = sbase + stage * kStageBytes;
          const uint64_t da = ptx::make_sdesc_sw128(sa, 16, 1024);
          const uint64_t db = ptx::make_sdesc_sw128(sa + kABytes, 16, 1024);
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k)
            ptx::umma_bf16_2cta(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          ptx::tc_commit_2cta(empty_bar + 8 * stage);  // frees the slot in both CTAs
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        ptx::tc_commit_2cta(acc_full + 8 * buf);
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps (both CTAs, own 128 rows)
    constexpr bool kFast = OutTraits<TOut>::kFast;
    constexpr int kBoxCols = 128 / static_cast<int>(sizeof(TOut));
    constexpr int kAccPerBox = (EPI == EPI_GLU) ? 2 * kBoxCols : kBoxCols;
    constexpr int kChunks = kAccPerBox / 32;
    constexpr int kBoxes = kBN / kAccPerBox;
    const int quarter = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row_in_tile = quarter * 32 + lane;
    uint8_t* stage_base = smem + kStagingOffset + (warp - 2) * 8192;
    // 32-bit shared-window addresses for the staging rows and the bias: through the rounded-up generic pointer the compiler
    // cannot prove the address space and emits generic LD.E / ST.E (long-scoreboard) for every access of the epilogue
    const uint32_t stage_a = ptx::smem_u32(stage_base), bias_a0 = ptx::smem_u32(smem + kBiasOffset);
    const uint32_t swz = static_cast<uint32_t>(lane & 7);
    uint32_t box_counter = 0;
    int it = 0;
    for (int tile = pair; tile < p.num_tiles; tile += num_pairs, ++it) {
      const int buf = it & 1;
      const int n_blk = tile % p.num_n_tiles;
      const int m_blk = 2 * (tile / p.num_n_tiles) + static_cast<int>(rank);  // this CTA's 128-row block
      const long long out_row = static_cast<long long>(m_blk) * kBlockM + row_in_tile;
      const bool row_ok = out_row < p.ep.M;
      const uint32_t bias_a = bias_a0 + buf * kBN * 4;
      {
        const int e = static_cast<int>(threadIdx.x) - 64;
        if (e < kBN) {
          const int col = n_blk * kBN + e;
          ptx::sts_f32(bias_a + 4 * e, (p.ep.bias != nullptr && col < p.ep.N) ? __ldg(p.ep.bias + col) : 0.f);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
      }
      const bool keep = row_ok ? epi_keep<EPI>(p.ep, out_row) : true;  // its load is in flight during the accumulator wait
      ptx::mbar_wait_a(acc_full + 8 * buf, (it >> 1) & 1);
      ptx::tc_fence_after();
      const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + buf * kBN;
#pragma unroll 1
      for (int box = half; box < kBoxes; box += kEpiWarps / 4) {
        const int acc_col0 = n_blk * kBN + box * kAccPerBox;
        if (acc_col0 >= p.ep.N) break;
        const int n_pass = (EPI == EPI_QKV && acc_col0 < p.ep.qkv_dp) ? 2 : 1;
#pragma unroll 1
        for (int pass = 0; pass < n_pass; ++pass) {
          uint8_t* sbuf = stage_base + (box_counter & 1u) * 4096;
          if (lane == 0) ptx::bulk_wait_read<1>();
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
                epi_compute<EPI, kFast>(p.ep, out_row, acc_col0 + ch * 32, acc, pass);
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
              constexpr int kPieces = (EPI == EPI_GLU) ? 2 : 4;
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
            ptx::bulk_commit();
          }
          ++box_counter;
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_leader(acc_empty + 8 * buf);  // one arrival per warp, on the leader's barrier
    }
    if (lane == 0) ptx::bulk_wait_read<0>();  // the staging boxes must outlive their reads
  }

  // neither CTA may retire (or free TMEM) while its partner can still read its shared memory or signal its barriers
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_2cta(tmem_base, kTmemCols);
  }
}

template <int EPI, typename TOut>
int launch_instance(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmO, const Tc2Params& p,
                    cudaStream_t st, std::string* err) {
  auto kern = gemm_tc2_kernel<EPI, TOut>;
  static bool configured[64] = {};
  static int max_pairs[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kTotal;
  cfg.stream = st;
  cfg.attrs = attr;
  if (!configured[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kTotal);
    if (e != cudaSuccess) {
      if (err) *err = std::string("cudaFuncSetAttribute(gemm_tc2): ") + cudaGetErrorString(e);
      return static_cast<int>(e);
    }
    int sms = 0, clusters = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cfg.gridDim = dim3(sms > 1 ? (sms / 2) * 2 : 2);
    cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&clusters, kern, &cfg) != cudaSuccess || clusters <= 0) {
      cudaGetLastError();
      clusters = sms / 2;
    }
    max_pairs[dev & 63] = clusters < sms / 2 ? clusters : sms / 2;
    if (max_pairs[dev & 63] < 1) max_pairs[dev & 63] = 1;
    configured[dev & 63] = true;
  }
  const int pairs = p.num_tiles < max_pairs[dev & 63] ? p.num_tiles : max_pairs[dev & 63];
  cfg.gridDim = dim3(2 * pairs);
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmO, p);
  if (e != cudaSuccess) {
    if (err) *err = std::string("gemm_tc2 launch: ") + cudaGetErrorString(e);
    return static_cast<int>(e);
  }
  return 0;
}

}  // namespace

bool gemm_tc2_supported(const GemmDesc& g) {
  return g.N % kBN == 0 && g.K % 8 == 0 && g.lda % 8 == 0 && g.ldw % 8 == 0 && g.M > kBlockM;
}

int launch_gemm_tc2(const GemmDesc& g, cudaStream_t st, std::string* err) {
  if (g.M <= 0 || g.N <= 0 || g.K <= 0) return 0;
  if (!gemm_tc2_supported(g)) {
    if (err) *err = "gemm_tc2: N must be a multiple of 256, K and the leading dimensions multiples of 8";
    return -1;
  }
  CUtensorMap tmA, tmB, tmO;
  {
    uint64_t dims[2] = {static_cast<uint64_t>(g.K), static_cast<uint64_t>(g.M)};
    uint64_t strides[1] = {static_cast<uint64_t>(g.lda) * 2};
    uint32_t box[2] = {kBlockK, kBlockM};
    if (!encode_tmap_bf16(&tmA, g.A, 2, dims, strides, box, err)) return -1;
  }
  {
    uint64_t dims[2] = {static_cast<uint64_t>(g.K), static_cast<uint64_t>(g.N)};
    uint64_t strides[1] = {static_cast<uint64_t>(g.ldw) * 2};
    uint32_t box[2] = {kBlockK, kBN / 2};
    if (!encode_tmap_bf16(&tmB, g.W, 2, dims, strides, box, err)) return -1;
  }
  Tc2Params p{};
  p.num_n_tiles = g.N / kBN;
  p.num_tiles = ((g.M + 2 * kBlockM - 1) / (2 * kBlockM)) * p.num_n_tiles;
  p.num_k_blocks = (g.K + kBlockK - 1) / kBlockK;
  p.ep = g.ep;
  p.ep.M = g.M;
  p.ep.N = g.N;
  {
    const bool f32 = !g.out_bf16 || g.epi == EPI_RESID;
    uint64_t cols = static_cast<uint64_t>(g.N);
    if (g.epi == EPI_QKV) cols = static_cast<uint64_t>(g.N) + g.ep.qkv_dp;
    if (g.epi == EPI_GLU) cols = static_cast<uint64_t>(g.N) / 2;
    if ((g.ep.ldo * (f32 ? 4 : 2)) % 16) {
      if (err) *err = "gemm_tc2: output leading dimension must be a multiple of 16 bytes";
      return -1;
    }
    uint64_t dims[2] = {cols, static_cast<uint64_t>(g.M)};
    uint64_t strides[1] = {static_cast<uint64_t>(g.ep.ldo) * (f32 ? 4 : 2)};
    uint32_t box[2] = {f32 ? 32u : 64u, 32u};
    if (!encode_tmap(&tmO, g.ep.out, f32, 2, dims, strides, box, err)) return -1;
  }
  switch (g.epi) {
    case EPI_LINEAR:
      return g.out_bf16 ? launch_instance<EPI_LINEAR, bf16>(tmA, tmB, tmO, p, st, err)
                        : launch_instance<EPI_LINEAR, float>(tmA, tmB, tmO, p, st, err);
    case EPI_SWISH:
      return launch_instance<EPI_SWISH, bf16>(tmA, tmB, tmO, p, st, err);
    case EPI_RELU:
      return launch_instance<EPI_RELU, bf16>(tmA, tmB, tmO, p, st, err);
    case EPI_RESID:
      return launch_instance<EPI_RESID, float>(tmA, tmB, tmO, p, st, err);
    case EPI_QKV:
      return launch_instance<EPI_QKV, bf16>(tmA, tmB, tmO, p, st, err);
    case EPI_GLU:
      return launch_instance<EPI_GLU, bf16>(tmA, tmB, tmO, p, st, err);
    default:
      if (err) *err = "gemm_tc2: unknown epilogue";
      return -1;
  }
}

}  // namespace cfb
