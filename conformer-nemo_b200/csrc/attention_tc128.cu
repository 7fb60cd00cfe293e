// Fused relative-position attention for heads 64 < dk <= 128 (padded to dkp = 128), sm_100a.  Same function as
// rel_attn_tc_kernel (attention_tc.cu); no T x T matrix ever reaches HBM:
//
//   ctx[i,:] = softmax_j( ((q_i+u).k_j + (q_i+v).p_{T-1+j-i}) / sqrt(dk) ) v_j        (multi_head_attention.py:195-210)
//
// The 64-wide layout does not carry over: Q+u | Q+v alone would take 128 TMEM columns, O_part (128 fp32 columns) no
// longer fits over S, and every operand tile doubles.  One CTA per (128-query tile, head, sequence); 256 threads, ONE
// softmax set, so there is no log-sum-exp merge:
//   TMEM  [  0, 64)  Q+v / 16 as the fp16 A operand of the G MMA (tcgen05.st by the thread that owns the row)
//         [ 64,128)  S = (Q+u) K^T of the current key tile (fp32)
//         [128,256)  O_part = P V of the current key tile (fp32, two 64-column MMAs)
//         [256,448)  ring of three 64-column blocks of G = (Q+v) Pband^T (fp16 accumulator, one column per element).
//                    Block g holds band rows T-1-i0-127 + 64 g .. +63 and lives in slot g % 3; key tile kt reads
//                    blocks kt..kt+2, so every block is computed ONCE and shared by three consecutive key tiles
//         [448,480)  probabilities P as a bf16 A operand (tcgen05.st), so P never touches smem
//   SMEM  Q+u (32 KB, TMA, the A operand of the S MMA: it has no room in TMEM), K ring (3 x 16 KB), V ring (2 x 16 KB),
//         band slots (3 x 16 KB, stored as two 64-column planes so that blocks 0..2 form one 192-row B operand), four
//         private shift rows (4 x 12.8 KB): 216 KB.  Every 128-wide tile is two 64-column SWIZZLE_128B boxes.
//   warp 0      TMA producer: Q+u, K and V tiles (separate rings: K is free after S, V only after P V) and band blocks
//   warp 1      S / P V issuer: S of tile kt+1 as soon as the softmax warps have read S of tile kt, then P V of tile kt,
//               so the next scores are ready when the current tile is folded
//   warp 2      G ring issuer
//   warp 3      idle (keeps the softmax warps on warp ids 4..7: tcgen05.ld reaches TMEM lanes 32 (warp % 4) ..)
//   warps 4..7  softmax (one query row per thread) with the running (max, sum, O[128]) in registers; O_part is folded
//               64 columns at a time.  rel_shift is the index remap of attention_tc.cu: a warp-uniform TMEM column
//               offset plus a per-lane offset applied through the private shift row; the window of tile kt+1 is
//               fetched while the P V MMA of tile kt runs.
// The position term runs on fp16 operands into an fp16 accumulator with (q + v) / 16 (attention_common.cuh), as at
// dk = 64.  The largest case of the headroom test multiplies q + v and p by 40: each product has standard deviation
// 40^2 = 1600, a sum of 128 of them 1600 sqrt(128) = 1.8 10^4, which is 1.1 10^3 after the division by 16; ~10^5 sums
// per head stay within about 4.5 sigma, 5 10^3, far below fp16's 65504 (dk = 64: 3.2 10^3).  A larger divisor would
// only cost precision of small scores.  Keys j >= len[b] are masked to -inf; query rows i >= len[b] and the pad columns dk..127 are written
// as exact zeros (linear_out reads them).
#include <cuda_fp16.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include "attention_common.cuh"
#include "common.cuh"
#include "ptx.cuh"

namespace cfb {
namespace {

constexpr int kBM = 128;   // queries per CTA
constexpr int kBN = 64;    // keys per tile
constexpr int kDK = 128;   // padded head dim
constexpr int kThreads = 256;
constexpr int kHalf = 64 * 64 * 2;          // one 64-row x 64-column box: 8 KB
constexpr int kQBytes = 2 * 2 * kHalf;      // 128 rows x 128 columns
constexpr int kKStages = 3, kVStages = 2;   // 16 KB per stage: [columns 0..63 | 64..127]
constexpr int kTileBytes = 2 * kHalf;
constexpr int kBandSlots = 3;               // = the G ring: slot g % 3 of both
constexpr int kPlaneBytes = kBandSlots * kHalf;  // band columns 0..63 of all slots, then 64..127
constexpr int kShiftPitch = 100;            // words per private shift row (see attention_tc.cu)
constexpr int kShiftBytes = 32 * kShiftPitch * 4;
constexpr int kOffQ = 0;
constexpr int kOffK = kOffQ + kQBytes;
constexpr int kOffV = kOffK + kKStages * kTileBytes;
constexpr int kOffBand = kOffV + kVStages * kTileBytes;
constexpr int kOffShift = kOffBand + 2 * kPlaneBytes;
constexpr int kOffBar = kOffShift + 4 * kShiftBytes;
constexpr int kBarBytes = 512;
constexpr int kSmemTotal = kOffBar + kBarBytes + 1024;
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColQv = 0, kColS = 64, kColO = 128, kColG = 256, kColP = 448;

struct AttnParams {
  const bf16* qkv;
  const int32_t* lens;
  bf16* ctx;
  int T, Dp, dk;
  const int4* tiles;  // packed batches: blockIdx.x -> (sequence, i0, first token row of its slot, rows in the slot)
  float scale_log2;   // log2(e) / sqrt(dk)
};

using namespace attn;  // shared device helpers (attention_common.cuh)

__global__ void __launch_bounds__(kThreads, 1)
rel_attn_tc128_kernel(const __grid_constant__ CUtensorMap tmKV, const __grid_constant__ CUtensorMap tmP,
                      const AttnParams p) {
  const int h = blockIdx.y;
  const int T = p.T;  // extent of the positional table (2T - 1 band rows)
  uint32_t tid;
  asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
  // through shuffles, as in attention_tc.cu: ptxas keeps a shuffle result instead of re-reading SR_TID.X in the loops
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(tid >> 5), 0);
  const int lane = __shfl_sync(0xffffffffu, static_cast<int>(tid & 31), static_cast<int>(tid & 31));

  extern __shared__ uint8_t smem_raw[];
  uint32_t sbase;
  asm volatile("mov.u32 %0, %1;" : "=r"(sbase) : "r"((ptx::smem_u32(smem_raw) + 1023u) & ~1023u));
  const uint32_t bar0 = sbase + kOffBar;
  const uint32_t qu_full = bar0 + 0;     // Q+u is in shared memory (TMA)
  const uint32_t qv_ready = bar0 + 8;    // Q+v is in TMEM (4 warp arrivals)
  const uint32_t s_full = bar0 + 16;     // S of the current key tile is in TMEM
  const uint32_t s_free = bar0 + 24;     // the softmax warps have read S: the next tile's S may be computed
  const uint32_t p_ready = bar0 + 32;    // P is in TMEM (and the previous O_part has been folded)
  const uint32_t o_full = bar0 + 40;     // O_part is in TMEM
  const uint32_t g_free = bar0 + 48;     // the G window of the current tile has been read out of the ring
  const uint32_t k_full = bar0 + 64;                     // [kKStages]
  const uint32_t k_empty = k_full + 8 * kKStages;        // [kKStages]
  const uint32_t v_full = k_empty + 8 * kKStages;        // [kVStages]
  const uint32_t v_empty = v_full + 8 * kVStages;        // [kVStages]
  const uint32_t band_full = v_empty + 8 * kVStages;     // [kBandSlots]
  const uint32_t band_empty = band_full + 8 * kBandSlots;  // [kBandSlots]
  const uint32_t g_full = band_empty + 8 * kBandSlots;   // [kBandSlots] G block in TMEM
  const uint32_t tmem_slot = g_full + 8 * kBandSlots;
  static_assert(64 + 8 * (2 * kKStages + 2 * kVStages + 3 * kBandSlots) + 8 <= kBarBytes, "barrier area");
  static_assert(kSmemTotal <= 227 * 1024, "shared memory budget");

  if (warp == 0) {
    if (lane == 0) {
      ptx::prefetch_tmap(&tmKV);
      ptx::prefetch_tmap(&tmP);
      ptx::mbar_init_a(qu_full, 1);
      ptx::mbar_init_a(qv_ready, 4);
      ptx::mbar_init_a(s_full, 1);
      ptx::mbar_init_a(s_free, 4);  // one elected arrival per softmax warp
      ptx::mbar_init_a(p_ready, 4);
      ptx::mbar_init_a(o_full, 1);
      ptx::mbar_init_a(g_free, 4);
      for (int s = 0; s < kKStages; ++s) {
        ptx::mbar_init_a(k_full + 8 * s, 1);
        ptx::mbar_init_a(k_empty + 8 * s, 1);
      }
      for (int s = 0; s < kVStages; ++s) {
        ptx::mbar_init_a(v_full + 8 * s, 1);
        ptx::mbar_init_a(v_empty + 8 * s, 1);
      }
      for (int s = 0; s < kBandSlots; ++s) {
        ptx::mbar_init_a(band_full + 8 * s, 1);
        ptx::mbar_init_a(band_empty + 8 * s, 1);
        ptx::mbar_init_a(g_full + 8 * s, 1);
      }
      ptx::fence_mbar_init();
    }
    __syncwarp();
  } else if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  pdl_launch_dependents();
  pdl_wait();
  // dense layout: sequence b owns rows [b T, b T + T); packed: the slot [rb, rb + S) of the tile table
  int i0 = blockIdx.x * kBM, b = blockIdx.z, S = T;
  long long rb = static_cast<long long>(b) * T;
  if (p.tiles != nullptr) {
    const int4 t = __ldg(p.tiles + blockIdx.x);
    b = t.x, i0 = t.y, rb = t.z, S = t.w;
  }
  const int len = min(p.lens[b], S);
  const bool active = i0 < len;  // otherwise the whole query tile is padding: the context rows are zero
  const int n_kt = active ? (len + kBN - 1) / kBN : 0;
  const int n_gb = n_kt + 2;  // G blocks 0 .. n_kt+1
  const int r0 = T - 1 - i0 - (kBM - 1);  // band row of G column 0 of block 0 (may be < 0: TMA zero-fills)

  // TMA loads of the 128-column tiles: two 64-column boxes each
  auto load_k = [&](int kt) {
    const int st = kt % kKStages;
    if (kt >= kKStages) ptx::mbar_wait_a(k_empty + 8 * st, ((kt / kKStages) & 1) ^ 1);
    ptx::mbar_arrive_expect_tx_a(k_full + 8 * st, kTileBytes);
    for (int c = 0; c < 2; ++c)
      ptx::tma_load_2d_a(sbase + kOffK + st * kTileBytes + c * kHalf, &tmKV, k_full + 8 * st, 2 * p.Dp + h * kDK + 64 * c,
                         static_cast<int>(rb) + kt * kBN);
  };
  auto load_v = [&](int kt) {
    const int st = kt % kVStages;
    if (kt >= kVStages) ptx::mbar_wait_a(v_empty + 8 * st, ((kt / kVStages) & 1) ^ 1);
    ptx::mbar_arrive_expect_tx_a(v_full + 8 * st, kTileBytes);
    for (int c = 0; c < 2; ++c)
      ptx::tma_load_2d_a(sbase + kOffV + st * kTileBytes + c * kHalf, &tmKV, v_full + 8 * st, 3 * p.Dp + h * kDK + 64 * c,
                         static_cast<int>(rb) + kt * kBN);
  };
  auto load_band = [&](int g) {
    const int slot = g % kBandSlots;
    if (g >= kBandSlots) ptx::mbar_wait_a(band_empty + 8 * slot, ((g / kBandSlots) & 1) ^ 1);
    ptx::mbar_arrive_expect_tx_a(band_full + 8 * slot, kTileBytes);
    for (int c = 0; c < 2; ++c)
      ptx::tma_load_2d_a(sbase + kOffBand + c * kPlaneBytes + slot * kHalf, &tmP, band_full + 8 * slot, h * kDK + 64 * c,
                         r0 + 64 * g);
  };

  uint32_t qw[64];  // softmax warps: this thread's row of Q+v, 128 bf16, fetched before the setup
  if (warp >= 4 && active) {
    const int i = i0 + (warp & 3) * 32 + lane;
    if (i < S) {
      const uint4* src = reinterpret_cast<const uint4*>(p.qkv + (rb + i) * (4 * p.Dp) + p.Dp + h * kDK);
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        const uint4 u = __ldg(src + c);
        qw[4 * c] = u.x, qw[4 * c + 1] = u.y, qw[4 * c + 2] = u.z, qw[4 * c + 3] = u.w;
      }
    } else {
#pragma unroll
      for (int c = 0; c < 64; ++c) qw[c] = 0u;
    }
  }

  if (warp == 0 && lane == 0 && active) {
    // the first loads only need their own barriers: issue them before the CTA-wide setup barrier.  Query rows past the
    // slot (or past the buffer: zero-filled) are computed but never written.
    ptx::mbar_arrive_expect_tx_a(qu_full, kQBytes);
    for (int c = 0; c < 2; ++c)
      for (int r = 0; r < 2; ++r)
        ptx::tma_load_2d_a(sbase + kOffQ + c * 2 * kHalf + r * kHalf, &tmKV, qu_full, h * kDK + 64 * c,
                           static_cast<int>(rb) + i0 + 64 * r);
    for (int g = 0; g < 3; ++g) load_band(g);
    load_k(0);
    load_v(0);
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  if (!active) {
    if (warp >= 4) {
      const int i = i0 + (warp & 3) * 32 + lane;
      if (i < S) {
        uint4* o = reinterpret_cast<uint4*>(p.ctx + (rb + i) * p.Dp + h * kDK);
#pragma unroll
        for (int c = 0; c < 16; ++c) o[c] = make_uint4(0, 0, 0, 0);
      }
    }
  } else if (warp == 0) {
    // ------------------------------------------------------------------------------------ TMA producer
    // in the order of need: K of tile kt (S runs one tile ahead), the band block of the window of tile kt, V of tile kt
    if (lane == 0) {
      for (int kt = 1; kt < n_kt; ++kt) {
        load_k(kt);
        load_band(kt + 2);
        load_v(kt);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------ S / P V issuer
    constexpr uint32_t idesc_s = ptx::make_idesc_bf16(kBM, kBN, 0, 0);
    constexpr uint32_t idesc_o = ptx::make_idesc_bf16(kBM, 64, 0, 1);  // B = V is MN-major (keys x dk rows)
    const uint32_t tS = tmem_base + kColS, tO = tmem_base + kColO, tP = tmem_base + kColP;
    auto issue_pv = [&](int t) {
      const int vs = t % kVStages;
      const uint32_t vst = sbase + kOffV + vs * kTileBytes;
      ptx::mbar_wait_a(v_full + 8 * vs, (t / kVStages) & 1);
      ptx::mbar_wait_a(p_ready, t & 1);
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {  // output columns 64 c .. 64 c + 63 from the c-th 64-column box of V
          const uint64_t dV = ptx::make_sdesc_sw128(vst + c * kHalf, 1024, 1024);
#pragma unroll
          for (int k = 0; k < kBN / 16; ++k)
            ptx::umma_bf16_ts(tO + 64 * c, tP + 8 * k, dV + static_cast<uint64_t>(k) * (2048 >> 4), idesc_o, k != 0);
        }
        ptx::tc_commit_a(o_full);
        ptx::tc_commit_a(v_empty + 8 * vs);
      }
      __syncwarp();
    };
    ptx::mbar_wait_a(qu_full, 0);
    for (int kt = 0; kt < n_kt; ++kt) {
      const int ks = kt % kKStages;
      const uint32_t kst = sbase + kOffK + ks * kTileBytes;
      ptx::mbar_wait_a(k_full + 8 * ks, (kt / kKStages) & 1);
      if (kt > 0) ptx::mbar_wait_a(s_free, (kt - 1) & 1);
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
#pragma unroll
        for (int k = 0; k < kDK / 16; ++k) {
          const uint64_t dQ = ptx::make_sdesc_sw128(sbase + kOffQ + (k >> 2) * 2 * kHalf, 16, 1024) + 2 * (k & 3);
          const uint64_t dK = ptx::make_sdesc_sw128(kst + (k >> 2) * kHalf, 16, 1024) + 2 * (k & 3);
          ptx::umma_bf16(tS, dQ, dK, idesc_s, k != 0);
        }
        ptx::tc_commit_a(s_full);
        ptx::tc_commit_a(k_empty + 8 * ks);
      }
      __syncwarp();
      if (kt > 0) issue_pv(kt - 1);
    }
    issue_pv(n_kt - 1);
  } else if (warp == 2) {
    // ------------------------------------------------------------------------------------ G ring issuer
    constexpr uint32_t idesc_g = make_idesc_f16_f16acc(kBM, 64);
    constexpr uint32_t idesc_g3 = make_idesc_f16_f16acc(kBM, 192);
    const uint32_t tQv = tmem_base + kColQv;
    const uint32_t band_base = sbase + kOffBand;
    ptx::mbar_wait_a(qv_ready, 0);
    // blocks 0..2 sit in consecutive band slots (per plane) and ring slots: one 192-wide MMA group
    ptx::mbar_wait_a(band_full + 0, 0);
    ptx::mbar_wait_a(band_full + 8, 0);
    ptx::mbar_wait_a(band_full + 16, 0);
    ptx::tc_fence_after();
    if (ptx::elect_one()) {
#pragma unroll
      for (int k = 0; k < kDK / 16; ++k) {
        const uint64_t dB = ptx::make_sdesc_sw128(band_base + (k >> 2) * kPlaneBytes, 16, 1024) + 2 * (k & 3);
        ptx::umma_bf16_ts(tmem_base + kColG, tQv + 8 * k, dB, idesc_g3, k != 0);
      }
      for (int s = 0; s < kBandSlots; ++s) {
        ptx::tc_commit_a(g_full + 8 * s);  // every ring slot's barrier advances one phase per block it receives
        ptx::tc_commit_a(band_empty + 8 * s);
      }
    }
    __syncwarp();
    for (int g = 3; g < n_gb; ++g) {
      const int bs = g % kBandSlots;
      ptx::mbar_wait_a(band_full + 8 * bs, (g / kBandSlots) & 1);
      // ring slot g%3 held block g-3, read by key tiles g-5 .. g-3 in this order: one wait for tile g-3.  The softmax
      // warps cannot be a phase further: their window of tile g-2 needs block g.
      ptx::mbar_wait_a(g_free, (g - 3) & 1);
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
#pragma unroll
        for (int k = 0; k < kDK / 16; ++k) {
          const uint64_t dB =
              ptx::make_sdesc_sw128(band_base + (k >> 2) * kPlaneBytes + bs * kHalf, 16, 1024) + 2 * (k & 3);
          ptx::umma_bf16_ts(tmem_base + kColG + bs * 64, tQv + 8 * k, dB, idesc_g, k != 0);
        }
        ptx::tc_commit_a(g_full + 8 * bs);
        ptx::tc_commit_a(band_empty + 8 * bs);
      }
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------------------------ softmax warps
    const int quarter = warp & 3;
    const int ii = quarter * 32 + lane;  // query row inside the tile == TMEM lane
    const int i = i0 + ii;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    const uint32_t tS = t_lane + kColS, tO = t_lane + kColO, tP = t_lane + kColP;

    // ---- this thread's row of (Q+v) / 16 as fp16 -> TMEM A operand of the G MMA (exact for a bf16 value inside fp16's range)
#pragma unroll
    for (int c = 0; c < 64; ++c) {
      const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&qw[c]));
      qw[c] = pack_f16x2(f.x * kGScaleInv, f.y * kGScaleInv);
    }
    ptx::tmem_st_x32(t_lane + kColQv, *reinterpret_cast<const uint32_t(*)[32]>(&qw[0]));
    ptx::tmem_st_x32(t_lane + kColQv + 32, *reinterpret_cast<const uint32_t(*)[32]>(&qw[32]));
    ptx::tc_wait_st();
    ptx::tc_fence_before();
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive_a(qv_ready);

    // rel_shift (attention_tc.cu): row ii needs window column (31 - lane) + jj of the 96 columns starting at
    // column 96 - 32 quarter of the concatenation of ring blocks kt, kt+1, kt+2
    const int sh = 31 - lane;
    const uint32_t shift_row = sbase + kOffShift + quarter * kShiftBytes + lane * 96 * 4 +
                               static_cast<uint32_t>(((lane >> 1) + 4 * (lane & 1)) & 7) * 16;
    const int wcol = 96 - 32 * quarter;

    auto fetch_window = [&](int kt) {
      ptx::mbar_wait_a(g_full + 8 * ((kt + 2) % kBandSlots), ((kt + 2) / kBandSlots) & 1);  // blocks complete in order
      ptx::tc_fence_after();
      uint32_t w[49];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int wc = wcol + 32 * c;
        const int blk = kt + (wc >> 6);
        ptx::tmem_ld_x16_pack16(t_lane + kColG + (blk % kBandSlots) * 64 + (wc & 63), &w[16 * c]);
      }
      ptx::tc_wait_ld();
      w[48] = 0u;
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_a(g_free);
      // odd shifts: move the row down by one half so that the halves (31 - lane) + 2 j, + 2 j + 1 share a word
      const uint32_t sel = (sh & 1) ? 0x5432u : 0x3210u;
#pragma unroll
      for (int m = 0; m < 48; ++m) w[m] = prmt(w[m], w[m + 1], sel);
#pragma unroll
      for (int q = 0; q < 12; ++q) ptx::sts128(shift_row + q * 16, w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
    };

    float o_acc[kDK];
#pragma unroll
    for (int c = 0; c < kDK; ++c) o_acc[c] = 0.f;
    float m_run = -INFINITY, l_run = 0.f;
    const float scale = p.scale_log2;

    fetch_window(0);
    for (int kt = 0; kt < n_kt; ++kt) {
      const int j0 = kt * kBN;
      uint32_t gw[32];
      lds_u32x32(shift_row + (sh >> 1) * 4, gw);
      ptx::mbar_wait_a(s_full, kt & 1);
      ptx::tc_fence_after();
      float sv[kBN];
      {
        uint32_t s0r[32], s1r[32];
        ptx::tmem_ld_x32(tS, s0r);
        ptx::tmem_ld_x32(tS + 32, s1r);
        ptx::tc_wait_ld();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_a(s_free);  // the next tile's S may be computed now
#pragma unroll
        for (int c = 0; c < 16; ++c) {  // s + 16 g, g an fp16 half of the packed window word
          ptx::fhfma_pair(gw[c], kGScaleH, __uint_as_float(s0r[2 * c]), __uint_as_float(s0r[2 * c + 1]), sv[2 * c], sv[2 * c + 1]);
          ptx::fhfma_pair(gw[16 + c], kGScaleH, __uint_as_float(s1r[2 * c]), __uint_as_float(s1r[2 * c + 1]), sv[32 + 2 * c],
                          sv[32 + 2 * c + 1]);
        }
      }
      if (j0 + kBN > len) {  // only the last key tile can contain masked keys
#pragma unroll
        for (int c = 0; c < kBN; ++c)
          if (j0 + c >= len) sv[c] = -INFINITY;
      }
      float mx4[4] = {sv[0], sv[1], sv[2], sv[3]};
#pragma unroll
      for (int c = 4; c < kBN; ++c) mx4[c & 3] = fmaxf(mx4[c & 3], sv[c]);
      const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      const float m_new = fmaxf(m_run, mx);  // finite: every tile holds at least one key j < len
      const float ms = m_new * scale;
      const float alpha = fast_exp2(fmaf(m_run, scale, -ms));
      float2 rs4[4] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
      const float2 scale2 = make_float2(scale, scale), nms2 = make_float2(-ms, -ms), alpha2 = make_float2(alpha, alpha);
      uint32_t pw[32];
#pragma unroll
      for (int m = 0; m < 32; ++m) {
        const float2 a = ptx::ffma2(make_float2(sv[2 * m], sv[2 * m + 1]), scale2, nms2);
        const float2 e = make_float2(fast_exp2(a.x), fast_exp2(a.y));
        rs4[m & 3] = ptx::fadd2(rs4[m & 3], e);
        pw[m] = prmt(__float_as_uint(e.x) + 0x8000u, __float_as_uint(e.y) + 0x8000u, 0x7632u);  // bf16, round half up
      }
      ptx::tmem_st_x32(tP, pw);
      const float2 rs2 = ptx::fadd2(ptx::fadd2(rs4[0], rs4[1]), ptx::fadd2(rs4[2], rs4[3]));
      l_run = fmaf(l_run, alpha, rs2.x + rs2.y);
      m_run = m_new;
      ptx::tc_wait_st();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_a(p_ready);
      // ---- the G window of the next tile, while the P V MMA runs
      if (kt + 1 < n_kt) fetch_window(kt + 1);
      // ---- o_acc = o_acc * alpha + O_part, 64 columns at a time
      ptx::mbar_wait_a(o_full, kt & 1);
      ptx::tc_fence_after();
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        uint32_t a0[32], a1[32];
        ptx::tmem_ld_x32(tO + 64 * hf, a0);
        ptx::tmem_ld_x32(tO + 64 * hf + 32, a1);
        ptx::tc_wait_ld();
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          float* oa = o_acc + 64 * hf;
          const float2 x = ptx::ffma2(make_float2(oa[2 * c], oa[2 * c + 1]), alpha2,
                                      make_float2(__uint_as_float(a0[2 * c]), __uint_as_float(a0[2 * c + 1])));
          const float2 y = ptx::ffma2(make_float2(oa[32 + 2 * c], oa[33 + 2 * c]), alpha2,
                                      make_float2(__uint_as_float(a1[2 * c]), __uint_as_float(a1[2 * c + 1])));
          oa[2 * c] = x.x, oa[2 * c + 1] = x.y, oa[32 + 2 * c] = y.x, oa[33 + 2 * c] = y.y;
        }
      }
      ptx::tc_fence_before();  // the next P store (p_ready) also tells the issuer that O_part has been read
    }

    // ---- context row: padded query rows and the pad columns dk..127 are exact zeros
    if (i < S) {
      const float inv = (i < len && l_run > 0.f) ? 1.f / l_run : 0.f;
      const bool valid = i < len;
      uint4* o = reinterpret_cast<uint4*>(p.ctx + (rb + i) * p.Dp + h * kDK);
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = (valid && 8 * c + e < p.dk) ? o_acc[8 * c + e] * inv : 0.f;
        o[c] = make_uint4(ptx::pack_bf16x2(v[0], v[1]), ptx::pack_bf16x2(v[2], v[3]), ptx::pack_bf16x2(v[4], v[5]),
                          ptx::pack_bf16x2(v[6], v[7]));
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace

int launch_attn_tc128(const AttnDesc& a, cudaStream_t st, std::string* err) {
  if ((a.tiles == nullptr && a.B <= 0) || a.T <= 0) return 0;
  if (a.dkp != kDK || a.dk < 1 || a.dk > kDK) {
    if (err) *err = "attn_tc128: padded head dim must be 128 and 1 <= dk <= 128";
    return -1;
  }
  const int Dp = a.H * kDK;
  const long long rows = a.tiles != nullptr ? a.rows : static_cast<long long>(a.B) * a.T;
  CUtensorMap tmKV, tmP;
  {
    // one 64-column x 64-row box serves Q+u (four boxes), K and V (two each)
    uint64_t dims[2] = {static_cast<uint64_t>(4 * Dp), static_cast<uint64_t>(rows)};
    uint64_t strides[1] = {static_cast<uint64_t>(4 * Dp) * 2};
    uint32_t box[2] = {64, 64};
    if (!encode_tmap_bf16(&tmKV, a.qkv, 2, dims, strides, box, err)) return -1;
  }
  const void* pos16 = attn_pos_f16(a, Dp, st);  // fp16 projections the G MMA reads (see attention_tc.cu)
  {
    uint64_t dims[2] = {static_cast<uint64_t>(Dp), static_cast<uint64_t>(2 * a.T - 1)};
    uint64_t strides[1] = {static_cast<uint64_t>(a.pos_f16 ? a.ld_pos : Dp) * 2};
    uint32_t box[2] = {64, 64};
    if (!encode_tmap_bf16(&tmP, pos16, 2, dims, strides, box, err)) return -1;
  }
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63]) {
    const cudaError_t e = cudaFuncSetAttribute(rel_attn_tc128_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTotal);
    if (e != cudaSuccess) {
      if (err) *err = std::string("cudaFuncSetAttribute(attn_tc128): ") + cudaGetErrorString(e);
      return static_cast<int>(e);
    }
    configured[dev & 63] = true;
  }
  AttnParams p;
  p.qkv = reinterpret_cast<const bf16*>(a.qkv);
  p.lens = a.lens;
  p.ctx = reinterpret_cast<bf16*>(a.ctx);
  p.T = a.T;
  p.Dp = Dp;
  p.dk = a.dk;
  p.tiles = a.tiles;
  p.scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(a.dk));
  dim3 grid((a.T + kBM - 1) / kBM, a.H, a.B);
  if (a.tiles != nullptr) grid = dim3(a.n_tiles, a.H, 1);
  const cudaError_t e = launch_pdl(rel_attn_tc128_kernel, grid, dim3(kThreads), kSmemTotal, st, tmKV, tmP, p);
  if (e != cudaSuccess) {
    if (err) *err = std::string("attn_tc128 launch: ") + cudaGetErrorString(e);
    return static_cast<int>(e);
  }
  return 0;
}

}  // namespace cfb
