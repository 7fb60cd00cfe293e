// Fused relative-position attention for sm_100a (flash-style; no T x T matrix ever reaches HBM).
//
//   ctx[i,:] = softmax_j( ((q_i+u).k_j + (q_i+v).p_{T-1+j-i}) / sqrt(dk) ) v_j        (multi_head_attention.py:195-210)
//
// One CTA per (128-query tile, head, sequence); 384 threads = 3 warpgroups (registers re-balanced with setmaxnreg).
// Everything a key tile needs from shared memory is read exactly once; the MMA A operands live in tensor memory:
//   TMEM  [  0, 64)  Q+u | Q+v as bf16 A operands (written once with tcgen05.st by the thread that owns the row)
//         [ 64,192)  per softmax set: S = (Q+u) K^T of the set's key tile, later overwritten by O_part = P V
//         [192,256)  per softmax set: probabilities P as a bf16 A operand (tcgen05.st), so P never touches smem
//         [256,512)  ring of four 64-column blocks of G = (Q+v) Pband^T.  Block g holds band rows
//                    T-1-i0-127 + 64 g .. +63; key tile kt reads blocks kt..kt+2, so every block is computed ONCE
//                    and shared by three consecutive key tiles (and by both softmax sets)
//   warp 0      TMA producer: K and V tiles (4-stage ring) and 64-row band blocks of linear_pos(pos_emb) (3 slots)
//   warps 1, 2  MMA issuers of softmax set 0 / 1: S, then O_part = P V once the set has stored its probabilities
//   warp 3      MMA issuer of the G ring
//   warps 4..11 two softmax sets of four warps (one query row per thread).  Set s owns key tiles s, s+2, ... with a
//               private running (max, sum, O); the sets ping-pong and are merged (log-sum-exp) at the end.
//               rel_shift is an index remap -- row ii needs G[ii][127-ii+jj] -- done as a warp-uniform TMEM column
//               offset plus a per-lane offset applied through a private shared-memory row holding the 96-column
//               window as packed fp16 pairs (conflict-free 16-byte stores, 4-byte loads; odd shifts are realigned
//               with one PRMT per word before the store).  The window of the set's NEXT tile is fetched while the
//               P V MMA of the current tile runs.
// Keys j >= len[b] are masked to -inf (the reference's -10000 underflows to exactly 0 for valid rows); query rows
// i >= len[b] are written as zeros (multi_head_attention.py:104-113, SURVEY.md 4.3).
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
constexpr int kDK = 64;    // padded head dim
constexpr int kThreads = 384;  // warpgroup 0: TMA + MMA issuers; warpgroups 1, 2: softmax sets 0, 1.  (The SMSP arbiter
                               // favours high warp ids: issuers placed ABOVE the softmax warps were measured to
                               // steal issue slots with their mbarrier polling, +15 % kernel time.)
constexpr int kKBytes = kBN * kDK * 2;     // 8 KB
constexpr int kKVStages = 4;               // K + V tiles, 16 KB per stage
constexpr int kKVBytes = 2 * kKBytes;
constexpr int kBandSlots = 3;              // 64-row band blocks in flight (each is consumed by exactly one MMA)
constexpr int kBlockBytes = 64 * kDK * 2;
constexpr int kGSlots = 4;                 // TMEM ring of G blocks
constexpr int kShiftPitch = 100;           // words per private shift row (96-column fp32 window + pad): 16-byte
                                           // stores and 4-byte loads at word offset (31 - lane) are conflict-free
constexpr int kShiftBytes = 32 * kShiftPitch * 4;
constexpr int kXPitch = 68;                // words per row of the end-of-kernel set exchange (m, l, O[64])
constexpr int kOffKV = 0;
constexpr int kOffBand = kOffKV + kKVStages * kKVBytes;
constexpr int kOffShift = kOffBand + kBandSlots * kBlockBytes;
constexpr int kOffBar = kOffShift + 8 * kShiftBytes;
constexpr int kBarBytes = 512;
constexpr int kSmemTotal = kOffBar + kBarBytes + 1024;
static_assert(4 * 32 * kXPitch * 4 <= kKVStages * kKVBytes, "set exchange must fit in the K/V ring");
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColQ = 0, kColS = 64, kColP = 192, kColG = 256;

struct AttnParams {
  const bf16* qkv;
  const int32_t* lens;
  bf16* ctx;
  int T, Dp;
  const int4* tiles;  // packed batches: blockIdx.x -> (sequence, i0, first token row of its slot, rows in the slot)
  float scale_log2;  // log2(e) / sqrt(dk)
};

using namespace attn;  // shared device helpers (attention_common.cuh)

__global__ void __launch_bounds__(kThreads, 1)
rel_attn_tc_kernel(const __grid_constant__ CUtensorMap tmKV, const __grid_constant__ CUtensorMap tmP,
                   const AttnParams p) {
  const int h = blockIdx.y;
  const int T = p.T;  // extent of the positional table (2T - 1 band rows)
  uint32_t tid;
  asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
  // Through a shuffle: ptxas rematerialises S2R SR_TID.X (tens of cycles) in front of the addresses that derive from the
  // warp and lane index -- several times per key tile in the softmax warps (ncu source page); a shuffle result it keeps.
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(tid >> 5), 0);
  const int lane = __shfl_sync(0xffffffffu, static_cast<int>(tid & 31), static_cast<int>(tid & 31));

  extern __shared__ uint8_t smem_raw[];
  // every shared-memory object is addressed through a 32-bit shared address derived once from this base
  // Laundered through a volatile mov: ptxas otherwise REMATERIALISES the base wherever it is short of registers, and the
  // recipe starts with S2R SR_CgaCtaId (tens of cycles) -- twice per key tile in the softmax warps (ncu source page).
  uint32_t sbase;
  asm volatile("mov.u32 %0, %1;" : "=r"(sbase) : "r"((ptx::smem_u32(smem_raw) + 1023u) & ~1023u));
  const uint32_t bar0 = sbase + kOffBar;
  const uint32_t qu_ready = bar0 + 0;    // Q+u is in TMEM (4 warp arrivals, softmax set 0)
  const uint32_t qv_ready = bar0 + 8;    // Q+v is in TMEM (4 warp arrivals, softmax set 1)
  const uint32_t sg_full = bar0 + 16;    // [2] per set: S of the set's current key tile is in TMEM
  const uint32_t s_free = bar0 + 32;     // [2] O_part folded: the S columns may be overwritten
  const uint32_t g_free = bar0 + 48;     // [2] per set: the G window of the set's tile has been read out of the ring
  const uint32_t p_ready = bar0 + 64;    // [2]
  const uint32_t o_full = bar0 + 80;     // [2]
  const uint32_t exp_done = bar0 + 96;   // [2] per set: the exponentials of the set's tile have issued
  const uint32_t kv_full = bar0 + 112;                   // [kKVStages]
  const uint32_t kv_empty = kv_full + 8 * kKVStages;     // [kKVStages]
  const uint32_t band_full = kv_empty + 8 * kKVStages;   // [kBandSlots]
  const uint32_t band_empty = band_full + 8 * kBandSlots;  // [kBandSlots]
  const uint32_t g_full = band_empty + 8 * kBandSlots;   // [kGSlots] G block in TMEM
  const uint32_t tmem_slot = g_full + 8 * kGSlots;
  static_assert(112 + 8 * (2 * kKVStages + 2 * kBandSlots + kGSlots) + 8 <= kBarBytes, "barrier area");
  static_assert(kSmemTotal <= 227 * 1024, "shared memory budget");

  // Barrier init and the TMEM allocation overlap the previous kernel's tail (programmatic dependent launch);
  // everything that reads global memory comes after pdl_wait().
  if (warp == 0) {
    if (lane == 0) {
      ptx::prefetch_tmap(&tmKV);
      ptx::prefetch_tmap(&tmP);
      ptx::mbar_init_a(qu_ready, 4);
      ptx::mbar_init_a(qv_ready, 4);
      for (int s = 0; s < kKVStages; ++s) {
        ptx::mbar_init_a(kv_full + 8 * s, 1);
        ptx::mbar_init_a(kv_empty + 8 * s, 1);
      }
      for (int s = 0; s < kBandSlots; ++s) {
        ptx::mbar_init_a(band_full + 8 * s, 1);
        ptx::mbar_init_a(band_empty + 8 * s, 1);
      }
      for (int s = 0; s < kGSlots; ++s) ptx::mbar_init_a(g_full + 8 * s, 1);
      for (int s = 0; s < 2; ++s) {
        ptx::mbar_init_a(sg_full + 8 * s, 1);
        ptx::mbar_init_a(s_free + 8 * s, 4);   // one elected arrival per softmax warp
        ptx::mbar_init_a(g_free + 8 * s, 4);
        ptx::mbar_init_a(p_ready + 8 * s, 4);
        ptx::mbar_init_a(o_full + 8 * s, 1);
        ptx::mbar_init_a(exp_done + 8 * s, 4);
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

  uint32_t qw[32];  // softmax warps: this thread's row of Q+u (set 0) / Q+v (set 1), 64 bf16, fetched before the setup
  if (warp >= 4 && active) {
    const int i = i0 + (warp & 3) * 32 + lane;
    if (i < S) {
      const uint4* src = reinterpret_cast<const uint4*>(p.qkv + (rb + i) * (4 * p.Dp) +
                                                        ((warp - 4) >> 2) * p.Dp + h * kDK);
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const uint4 u = __ldg(src + c);
        qw[4 * c] = u.x, qw[4 * c + 1] = u.y, qw[4 * c + 2] = u.z, qw[4 * c + 3] = u.w;
      }
    } else {
#pragma unroll
      for (int c = 0; c < 32; ++c) qw[c] = 0u;
    }
  }

  if (warp == 0 && lane == 0 && active) {
    // the first loads only need their own barriers: issue them before the CTA-wide setup barrier
    const int r0 = T - 1 - i0 - (kBM - 1);  // band row of G column 0 of block 0 (may be < 0: TMA zero-fills)
#pragma unroll
    for (int g = 0; g < 3; ++g) {
      ptx::mbar_arrive_expect_tx_a(band_full + 8 * g, kBlockBytes);
      ptx::tma_load_2d_a(sbase + kOffBand + g * kBlockBytes, &tmP, band_full + 8 * g, h * kDK, r0 + 64 * g);
    }
    ptx::mbar_arrive_expect_tx_a(kv_full, kKVBytes);
    ptx::tma_load_2d_a(sbase + kOffKV, &tmKV, kv_full, 2 * p.Dp + h * kDK, static_cast<int>(rb));
    ptx::tma_load_2d_a(sbase + kOffKV + kKBytes, &tmKV, kv_full, 3 * p.Dp + h * kDK, static_cast<int>(rb));
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  if (!active) {
    if (warp >= 4 && warp < 8) {
      const int i = i0 + (warp & 3) * 32 + lane;
      if (i < S) {
        uint4* o = reinterpret_cast<uint4*>(p.ctx + (rb + i) * p.Dp + h * kDK);
#pragma unroll
        for (int c = 0; c < 8; ++c) o[c] = make_uint4(0, 0, 0, 0);
      }
    }
  } else if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;" ::: "memory");
    if (warp == 0) {
      // ---------------------------------------------------------------------------------- TMA producer
      if (lane == 0) {
        const int r0 = T - 1 - i0 - (kBM - 1);
        auto load_band_block = [&](int g) {
          if (g >= n_gb) return;
          const int slot = g % kBandSlots, use = g / kBandSlots;
          ptx::mbar_wait_a(band_empty + 8 * slot, (use & 1) ^ 1);
          ptx::mbar_arrive_expect_tx_a(band_full + 8 * slot, kBlockBytes);
          ptx::tma_load_2d_a(sbase + kOffBand + slot * kBlockBytes, &tmP, band_full + 8 * slot, h * kDK, r0 + 64 * g);
        };
        load_band_block(3);
        for (int kt = 1; kt < n_kt; ++kt) {
          const int st = kt % kKVStages, use = kt / kKVStages;
          ptx::mbar_wait_a(kv_empty + 8 * st, (use & 1) ^ 1);
          ptx::mbar_arrive_expect_tx_a(kv_full + 8 * st, kKVBytes);
          const uint32_t dst = sbase + kOffKV + st * kKVBytes;
          ptx::tma_load_2d_a(dst, &tmKV, kv_full + 8 * st, 2 * p.Dp + h * kDK, static_cast<int>(rb) + kt * kBN);
          ptx::tma_load_2d_a(dst + kKBytes, &tmKV, kv_full + 8 * st, 3 * p.Dp + h * kDK, static_cast<int>(rb) + kt * kBN);
          load_band_block(kt + 3);
        }
      }
    } else if (warp == 1 || warp == 2) {
      // ---------------------------------------------------------------------------------- S / PV issuer of a set
      // Warp-uniform control flow (all lanes wait, one elected lane issues): addresses and descriptors stay in
      // uniform registers, which keeps the wait -> first-MMA latency on the softmax critical path short.
      const int s = warp - 1;
      constexpr uint32_t idesc_s = ptx::make_idesc_bf16(kBM, kBN, 0, 0);
      constexpr uint32_t idesc_o = ptx::make_idesc_bf16(kBM, kDK, 0, 1);  // B = V is MN-major (keys x dk rows)
      const uint32_t tQu = tmem_base + kColQ;
      const uint32_t tS = tmem_base + kColS + s * 64;
      const uint32_t tP = tmem_base + kColP + s * 32;
      ptx::mbar_wait_a(qu_ready, 0);
      ptx::tc_fence_after();
      int it = 0;
      for (int kt = s; kt < n_kt; kt += 2, ++it) {
        const int kvs = kt % kKVStages;
        const uint32_t st = sbase + kOffKV + kvs * kKVBytes;
        const uint64_t dK = ptx::make_sdesc_sw128(st, 16, 1024);
        // V tile: 64 keys (K of this MMA) x 64 dk (N), 128-byte rows along N -> MN-major, 8-key groups 1 KB apart
        const uint64_t dV = ptx::make_sdesc_sw128(st + kKBytes, 1024, 1024);
        ptx::mbar_wait_a(kv_full + 8 * kvs, (kt / kKVStages) & 1);
        ptx::mbar_wait_a(s_free + 8 * s, (it & 1) ^ 1);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
#pragma unroll
          for (int k = 0; k < kDK / 16; ++k) ptx::umma_bf16_ts(tS, tQu + 8 * k, dK + 2 * k, idesc_s, k != 0);
          ptx::tc_commit_a(sg_full + 8 * s);
        }
        __syncwarp();
        // ---- O_part = P V once the set has stored its probabilities (P is a TMEM A operand: 8 columns per K=16)
        ptx::mbar_wait_a(p_ready + 8 * s, it & 1);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
#pragma unroll
          for (int k = 0; k < kBN / 16; ++k)
            ptx::umma_bf16_ts(tS, tP + 8 * k, dV + static_cast<uint64_t>(k) * (2048 >> 4), idesc_o, k != 0);
          ptx::tc_commit_a(o_full + 8 * s);
          ptx::tc_commit_a(kv_empty + 8 * kvs);
        }
        __syncwarp();
      }
    } else {
      // ---------------------------------------------------------------------------------- G ring issuer
      constexpr uint32_t idesc_g = make_idesc_f16_f16acc(kBM, 64);
      constexpr uint32_t idesc_g3 = make_idesc_f16_f16acc(kBM, 192);
      const uint32_t tQv = tmem_base + kColQ + 32;
      const uint32_t band_base = sbase + kOffBand;
      ptx::mbar_wait_a(qv_ready, 0);
      // blocks 0..2 sit in consecutive band slots and ring slots: one 192-wide MMA group
      ptx::mbar_wait_a(band_full + 0, 0);
      ptx::mbar_wait_a(band_full + 8, 0);
      ptx::mbar_wait_a(band_full + 16, 0);
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        const uint64_t dB = ptx::make_sdesc_sw128(band_base, 16, 1024);
#pragma unroll
        for (int k = 0; k < kDK / 16; ++k)
          ptx::umma_bf16_ts(tmem_base + kColG, tQv + 8 * k, dB + 2 * k, idesc_g3, k != 0);
        ptx::tc_commit_a(g_full + 0);  // every ring slot's barrier advances one phase per block it receives
        ptx::tc_commit_a(g_full + 8);
        ptx::tc_commit_a(g_full + 16);
        ptx::tc_commit_a(band_empty + 0);
        ptx::tc_commit_a(band_empty + 8);
        ptx::tc_commit_a(band_empty + 16);
      }
      __syncwarp();
      for (int g = 3; g < n_gb; ++g) {
        const int bs = g % kBandSlots;
        const uint64_t dB = ptx::make_sdesc_sw128(band_base + bs * kBlockBytes, 16, 1024);
        const uint32_t tG = tmem_base + kColG + (g % kGSlots) * 64;
        ptx::mbar_wait_a(band_full + 8 * bs, (g / kBandSlots) & 1);
        // ring slot g%4 held block g-4, read by key tiles g-6, g-5, g-4.  Tile g-5 (the other set's) was waited
        // for at step g-1 and tile g-6 precedes g-4 in its set, so one wait per step covers all three readers
        // (waiting again for g-5 here could alias: that set may already be two phases further).
        if (g >= 4 && g - 4 < n_kt) ptx::mbar_wait_a(g_free + 8 * ((g - 4) & 1), ((g - 4) >> 1) & 1);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
#pragma unroll
          for (int k = 0; k < kDK / 16; ++k) ptx::umma_bf16_ts(tG, tQv + 8 * k, dB + 2 * k, idesc_g, k != 0);
          ptx::tc_commit_a(g_full + 8 * (g % kGSlots));
          ptx::tc_commit_a(band_empty + 8 * bs);
        }
        __syncwarp();
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;" ::: "memory");
    // ---------------------------------------------------------------------------------- softmax warps
    const int quarter = warp & 3;
    const int set = (warp - 4) >> 2;
    const int ii = quarter * 32 + lane;  // query row inside the tile == TMEM lane
    const int i = i0 + ii;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    const uint32_t tS = t_lane + kColS + set * 64;
    const uint32_t tP = t_lane + kColP + set * 32;

    // ---- this thread's row of Q+u (set 0) or Q+v (set 1) -> TMEM A operand
    if (set == 1) {  // the G MMA takes fp16 operands: (q + v) / 16 as fp16 (exact for a bf16 value inside fp16's range)
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&qw[c]));
        qw[c] = pack_f16x2(f.x * kGScaleInv, f.y * kGScaleInv);
      }
    }
    ptx::tmem_st_x32(t_lane + kColQ + set * 32, qw);
    ptx::tc_wait_st();
    ptx::tc_fence_before();
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive_a(set == 0 ? qu_ready : qv_ready);

    // rel_shift: row ii needs window column (31 - lane) + jj of the 96 columns starting at ring column
    // 64 kt + 96 - 32 quarter.  The window goes through a private fp32 shared-memory row: stored with 16-byte
    // stores while the P V MMA of the previous tile runs, read back at word offset 31 - lane when S arrives.
    const int sh = 31 - lane;
    // 48 packed words per row, pitch 96 words plus a 16-byte skew ((lane / 2 + 4 (lane & 1)) mod 8) that keeps both the
    // 16-byte stores and the 4-byte loads at word offset (31 - lane) / 2 conflict-free
    const uint32_t shift_row = sbase + kOffShift + (warp - 4) * kShiftBytes + lane * 96 * 4 +
                               static_cast<uint32_t>(((lane >> 1) + 4 * (lane & 1)) & 7) * 16;
    const int wcol = 96 - 32 * quarter;  // window start inside the concatenation of ring blocks kt, kt+1, kt+2

    auto fetch_window = [&](int kt) {
      ptx::mbar_wait_a(g_full + 8 * ((kt + 2) % kGSlots), ((kt + 2) / kGSlots) & 1);  // blocks complete in order
      ptx::tc_fence_after();
      uint32_t w[49];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int wc = wcol + 32 * c;
        const int blk = kt + (wc >> 6);
        ptx::tmem_ld_x16_pack16(t_lane + kColG + (blk % kGSlots) * 64 + (wc & 63), &w[16 * c]);
      }
      ptx::tc_wait_ld();
      w[48] = 0u;
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_a(g_free + 8 * set);
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

    if (set < n_kt) fetch_window(set);
    int it = 0;
    for (int kt = set; kt < n_kt; kt += 2, ++it) {
      const int j0 = kt * kBN;
      // the shifted window row was stored a whole P V MMA ago: read it while the S MMA of this tile is still in flight
      uint32_t gw[32];
      lds_u32x32(shift_row + (sh >> 1) * 4, gw);
      ptx::mbar_wait_a(sg_full + 8 * set, it & 1);
      ptx::tc_fence_after();
      float sv[kBN];
      {
        uint32_t s0r[32], s1r[32];
        ptx::tmem_ld_x32(tS, s0r);
        ptx::tmem_ld_x32(tS + 32, s1r);
        ptx::tc_wait_ld();
#pragma unroll
        for (int c = 0; c < 16; ++c) {  // s + 16 g, g an fp16 half of the packed window word (FHFMA: no conversion)
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
      // The exponentials of consecutive key tiles take turns on the MUFU pipe (tile kt after tile kt-1): the two
      // sets then stay in anti-phase, one in its MUFU phase while the other is in its shared-memory / TMEM phases,
      // instead of drifting into lock-step and halving each other's throughput in every phase.
      if (kt > 0) ptx::mbar_wait_a(exp_done + 8 * (set ^ 1), (set == 0 ? it - 1 : it) & 1);
      float mx4[4] = {sv[0], sv[1], sv[2], sv[3]};  // four independent chains instead of one 64-deep one
#pragma unroll
      for (int c = 4; c < kBN; ++c) mx4[c & 3] = fmaxf(mx4[c & 3], sv[c]);
      const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      const float m_new = fmaxf(m_run, mx);  // finite: every tile holds at least one key j < len
      const float ms = m_new * scale;
      const float alpha = fast_exp2(fmaf(m_run, scale, -ms));
      // two fp32 lanes per instruction where the math allows (FFMA2 / FADD2, ptx.cuh): these warps are bound by the
      // length of their instruction stream
      float2 rs4[4] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
      const float2 scale2 = make_float2(scale, scale), nms2 = make_float2(-ms, -ms), alpha2 = make_float2(alpha, alpha);
      uint32_t pw[32];
#pragma unroll
      for (int m = 0; m < 32; ++m) {
        const float2 a = ptx::ffma2(make_float2(sv[2 * m], sv[2 * m + 1]), scale2, nms2);
        const float2 e = make_float2(fast_exp2(a.x), fast_exp2(a.y));
        rs4[m & 3] = ptx::fadd2(rs4[m & 3], e);
        // bf16 pair without the conversion unit (it shares the MUFU pipe): round half up with integer adds, one PRMT
        pw[m] = prmt(__float_as_uint(e.x) + 0x8000u, __float_as_uint(e.y) + 0x8000u, 0x7632u);
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_a(exp_done + 8 * set);
      ptx::tmem_st_x32(tP, pw);
      const float2 rs2 = ptx::fadd2(ptx::fadd2(rs4[0], rs4[1]), ptx::fadd2(rs4[2], rs4[3]));
      const float rsum = rs2.x + rs2.y;
      l_run = fmaf(l_run, alpha, rsum);
      m_run = m_new;
      ptx::tc_wait_st();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_a(p_ready + 8 * set);
      // ---- the G window of this set's next tile, while the P V MMA runs
      if (kt + 2 < n_kt) fetch_window(kt + 2);
      // ---- o_acc = o_acc * alpha + O_part (the S columns of this set)
      ptx::mbar_wait_a(o_full + 8 * set, it & 1);
      ptx::tc_fence_after();
      {
        uint32_t a0[32], a1[32];
        ptx::tmem_ld_x32(tS, a0);
        ptx::tmem_ld_x32(tS + 32, a1);
        ptx::tc_wait_ld();
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          const float2 x = ptx::ffma2(make_float2(o_acc[2 * c], o_acc[2 * c + 1]), alpha2,
                                      make_float2(__uint_as_float(a0[2 * c]), __uint_as_float(a0[2 * c + 1])));
          const float2 y = ptx::ffma2(make_float2(o_acc[32 + 2 * c], o_acc[33 + 2 * c]), alpha2,
                                      make_float2(__uint_as_float(a1[2 * c]), __uint_as_float(a1[2 * c + 1])));
          o_acc[2 * c] = x.x, o_acc[2 * c + 1] = x.y, o_acc[32 + 2 * c] = y.x, o_acc[33 + 2 * c] = y.y;
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_a(s_free + 8 * set);  // the S columns may now receive the next tile's scores
    }

    // ---- merge the two sets (log-sum-exp) and write the context rows.  Every MMA of the CTA has completed once
    // both sets are past their last o_full wait, so the K/V ring can carry the exchange (16-byte accesses,
    // 17-quad row pitch: conflict-free).
    asm volatile("bar.sync 1, 256;" ::: "memory");
    const uint32_t xrow = sbase + kOffKV + ii * kXPitch * 4;
    if (set == 1) {
      ptx::sts128(xrow, __float_as_uint(m_run), __float_as_uint(l_run), 0u, 0u);
#pragma unroll
      for (int c = 0; c < kDK / 4; ++c)
        ptx::sts128(xrow + 16 + 16 * c, __float_as_uint(o_acc[4 * c]), __float_as_uint(o_acc[4 * c + 1]),
                    __float_as_uint(o_acc[4 * c + 2]), __float_as_uint(o_acc[4 * c + 3]));
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (set == 0) {
      const float4 ml = lds_f32x4(xrow);
      const float m1 = ml.x, l1 = ml.y;
      const float m = fmaxf(m_run, m1);  // set 0 always owns key tile 0, so m is finite
      const float w0 = fast_exp2((m_run - m) * scale), w1 = fast_exp2((m1 - m) * scale);
      const float l = l_run * w0 + l1 * w1;
      const float inv = (i < len && l > 0.f) ? 1.f / l : 0.f;  // padded query rows -> zeros
      const float c0 = w0 * inv, c1 = w1 * inv;
      if (i < S) {
        uint4* o = reinterpret_cast<uint4*>(p.ctx + (rb + i) * p.Dp + h * kDK);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 x0 = lds_f32x4(xrow + 16 + 32 * c), x1 = lds_f32x4(xrow + 32 + 32 * c);
          uint4 u;
          u.x = ptx::pack_bf16x2(fmaf(o_acc[8 * c + 0], c0, x0.x * c1), fmaf(o_acc[8 * c + 1], c0, x0.y * c1));
          u.y = ptx::pack_bf16x2(fmaf(o_acc[8 * c + 2], c0, x0.z * c1), fmaf(o_acc[8 * c + 3], c0, x0.w * c1));
          u.z = ptx::pack_bf16x2(fmaf(o_acc[8 * c + 4], c0, x1.x * c1), fmaf(o_acc[8 * c + 5], c0, x1.y * c1));
          u.w = ptx::pack_bf16x2(fmaf(o_acc[8 * c + 6], c0, x1.z * c1), fmaf(o_acc[8 * c + 7], c0, x1.w * c1));
          o[c] = u;
        }
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

// The G MMA reads fp16 positional projections.  cfb_forward converts its whole `pos` buffer once per call, in place
// (launch_bf16_to_f16_inplace) and says so (pos_f16); the kernel-level entry point cfb_op_rel_attention takes bf16 like every
// other operand and gets a copy here: a lazily grown scratch buffer -- that path allocates, the forward does not.
const void* attn_pos_f16(const AttnDesc& a, int Dp, cudaStream_t st) {
  if (a.pos_f16) return a.pos;
  static void* scratch[64] = {};
  static size_t elems[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  const size_t need = static_cast<size_t>(2 * a.T - 1) * Dp;
  if (elems[dev & 63] < need) {
    if (scratch[dev & 63]) cudaFree(scratch[dev & 63]);
    cudaMalloc(&scratch[dev & 63], need * 2);
    elems[dev & 63] = need;
  }
  launch_bf16_to_f16(a.pos, a.ld_pos, scratch[dev & 63], 2 * a.T - 1, Dp, st);
  return scratch[dev & 63];
}

int launch_attn_tc(const AttnDesc& a, cudaStream_t st, std::string* err) {
  if ((a.tiles == nullptr && a.B <= 0) || a.T <= 0) return 0;
  if (a.dkp == 128) return launch_attn_tc128(a, st, err);  // no persistent form: CFB_ATTN_PERSIST does not apply
  if (a.dkp != kDK) {
    if (err) *err = "attn_tc: padded head dim must be 64 or 128";
    return -1;
  }
  {
    // persistent form (attention_tcp.cu).  Measured (r02t): 256 x 100 frames x 4 heads 48.3 -> 43.3 us, 32 x 500 x 8
    // 93.3 -> 92.1 us, 1 x 7500 x 8 477 -> 504 us: it removes the per-CTA setup, which matters for short sequences; the
    // per-item time is set by the softmax warps' serial work either way.  CFB_ATTN_PERSIST=1 / 0 forces.
    const char* pv = getenv("CFB_ATTN_PERSIST");
    // packed batches: the tiles of one launch differ widely in length, which the hardware's dynamic CTA scheduling
    // absorbs and a static item walk does not -- per-item form unless forced
    const bool want = pv != nullptr ? atoi(pv) != 0 : (a.tiles == nullptr && a.T <= 512);
    if (want) return launch_attn_tcp(a, st, err);
  }
  const int Dp = a.H * a.dkp;
  const long long rows = a.tiles != nullptr ? a.rows : static_cast<long long>(a.B) * a.T;
  CUtensorMap tmKV, tmP;
  {
    uint64_t dims[2] = {static_cast<uint64_t>(4 * Dp), static_cast<uint64_t>(rows)};
    uint64_t strides[1] = {static_cast<uint64_t>(4 * Dp) * 2};
    uint32_t boxk[2] = {kDK, kBN};
    if (!encode_tmap_bf16(&tmKV, a.qkv, 2, dims, strides, boxk, err)) return -1;
  }
  const void* pos16 = attn_pos_f16(a, Dp, st);  // fp16 copy of the projections the G MMA reads (in place in the engine's forward)
  {
    // 2-byte elements: the number format is the MMA's business, not the tensor map's
    uint64_t dims[2] = {static_cast<uint64_t>(Dp), static_cast<uint64_t>(2 * a.T - 1)};
    uint64_t strides[1] = {static_cast<uint64_t>(a.pos_f16 ? a.ld_pos : Dp) * 2};
    uint32_t box[2] = {kDK, 64};
    if (!encode_tmap_bf16(&tmP, pos16, 2, dims, strides, box, err)) return -1;
  }
  static bool configured[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63]) {
    const cudaError_t e = cudaFuncSetAttribute(rel_attn_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTotal);
    if (e != cudaSuccess) {
      if (err) *err = std::string("cudaFuncSetAttribute(attn_tc): ") + cudaGetErrorString(e);
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
  p.tiles = a.tiles;
  p.scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(a.dk));
  dim3 grid((a.T + kBM - 1) / kBM, a.H, a.B);
  if (a.tiles != nullptr) grid = dim3(a.n_tiles, a.H, 1);
  const cudaError_t e = launch_pdl(rel_attn_tc_kernel, grid, dim3(kThreads), kSmemTotal, st, tmKV, tmP, p);
  if (e != cudaSuccess) {
    if (err) *err = std::string("attn_tc launch: ") + cudaGetErrorString(e);
    return static_cast<int>(e);
  }
  return 0;
}

}  // namespace cfb
