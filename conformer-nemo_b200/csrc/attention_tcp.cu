// PERSISTENT form of the fused relative-position attention of attention_tc.cu (same math, same warp roles, same TMEM
// map): one CTA per SM walks over (query tile, head, sequence) items, and every pipeline -- K/V ring, band slots, the
// G ring in TMEM, the per-set S / P / O hand-shakes -- keeps running across items (ring indices and mbarrier phases are
// continuous), so the TMA producer and the MMA issuers are already working on the next item while the softmax warps
// merge and write the current one, and barrier init + TMEM allocation happen once per SM instead of once per item.
// attention_tc.cu's per-item prologue (lens -> Q fetch -> operand store -> first G blocks: 5.8 k cycles) and merge
// (3.1 k) were 35 % of a CTA's 25.2 k cycles at T' = 500 (profiles/r02r_attention_trace.log).
//
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
constexpr int kOffX = kOffBar + kBarBytes;  // set exchange (m, l, O[64]) x 128 rows: its own buffer (the K/V ring is busy)
constexpr int kItemCap = 64;                // work items of this CTA decoded once into shared memory (32 B each)
constexpr int kOffItems = kOffX + 4 * 32 * kXPitch * 4;
constexpr int kSmemTotal = kOffItems + kItemCap * 32 + 1024;
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColQ = 0, kColS = 64, kColP = 192, kColG = 256;

struct AttnPParams {
  const bf16* qkv;
  const int32_t* lens;
  bf16* ctx;
  int T, Dp, H;
  int n_qt;          // query tiles per sequence (dense layout) / query tiles in the tile table (packed)
  int n_items;       // B * H * n_qt, query tile fastest (CTAs that share K / V / band rows run side by side)
  const int4* tiles; // packed batches: (sequence, i0, first token row of the slot, rows in the slot); items = n_qt x H
  float scale_log2;  // log2(e) / sqrt(dk)
};

using namespace attn;  // shared device helpers (attention_common.cuh)

__global__ void __launch_bounds__(kThreads, 1)
rel_attn_tcp_kernel(const __grid_constant__ CUtensorMap tmKV, const __grid_constant__ CUtensorMap tmP,
                    const AttnPParams p) {
  const int T = p.T;
  uint32_t tid;
  asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
  // Through a shuffle: ptxas rematerialises S2R SR_TID.X (tens of cycles) in front of the addresses that derive from the
  // warp and lane index -- several times per key tile in the softmax warps (ncu source page); a shuffle result it keeps.
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(tid >> 5), 0);
  const int lane = __shfl_sync(0xffffffffu, static_cast<int>(tid & 31), static_cast<int>(tid & 31));

  extern __shared__ uint8_t smem_raw[];
  // Laundered through a volatile mov: ptxas otherwise REMATERIALISES the base wherever it is short of registers, and the
  // recipe starts with S2R SR_CgaCtaId (tens of cycles) -- twice per key tile in the softmax warps (ncu source page).
  uint32_t sbase;
  asm volatile("mov.u32 %0, %1;" : "=r"(sbase) : "r"((ptx::smem_u32(smem_raw) + 1023u) & ~1023u));
  const uint32_t bar0 = sbase + kOffBar;
  const uint32_t qu_ready = bar0 + 0;    // Q+u of the current item is in TMEM (4 warp arrivals, softmax set 0)
  const uint32_t qv_ready = bar0 + 8;    // Q+v (softmax set 1)
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
  const uint32_t role_sync = tmem_slot + 8;  // the three MMA issuer warps have started the current item
  static_assert(112 + 8 * (2 * kKVStages + 2 * kBandSlots + kGSlots) + 16 <= kBarBytes, "barrier area");
  static_assert(kSmemTotal <= 227 * 1024, "shared memory budget");

  if (warp == 0) {
    if (lane == 0) {
      ptx::prefetch_tmap(&tmKV);
      ptx::prefetch_tmap(&tmP);
      ptx::mbar_init_a(qu_ready, 4);
      ptx::mbar_init_a(qv_ready, 4);
      ptx::mbar_init_a(role_sync, 3);
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
        ptx::mbar_init_a(s_free + 8 * s, 4);
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
  // item -> (query tile, head, sequence) and the tile counts every role derives identically
  struct Item {
    int i0, h, b, len, n_kt, n_gb;
    int rb, S;  // first token row and row count of the sequence (dense: b T and T; packed: its slot)
    bool active;
  };
  auto finish = [](Item& it) {
    it.active = it.i0 < it.len;  // otherwise the whole query tile is padding: the context rows are zero
    it.n_kt = it.active ? (it.len + kBN - 1) / kBN : 0;
    it.n_gb = it.active ? it.n_kt + 2 : 0;
  };
  auto decode_direct = [&](int item) {
    Item it;
    const int qt = item % p.n_qt;
    const int r = item / p.n_qt;
    if (p.tiles != nullptr) {
      const int4 t = __ldg(p.tiles + qt);
      it.h = r;
      it.b = t.x, it.i0 = t.y, it.rb = t.z, it.S = t.w;
    } else {
      it.h = r % p.H;
      it.b = r / p.H;
      it.i0 = qt * kBM;
      it.rb = it.b * T;
      it.S = T;
    }
    it.len = min(__ldg(p.lens + it.b), it.S);
    finish(it);
    return it;
  };
  const int item0 = blockIdx.x, item_step = gridDim.x;
  const int n_mine = item0 < p.n_items ? (p.n_items - item0 + item_step - 1) / item_step : 0;
  const uint32_t item_tab = sbase + kOffItems;

  pdl_launch_dependents();
  pdl_wait();
  // Every role walks the same item list; the divisions and the dependent length load of a decode sat on the softmax
  // warps' path between items (ncu source page: long-scoreboard stalls in the merge / write-back part).  The first
  // kItemCap items are decoded here once, in parallel, with the "is any later item active" answer the exchange barrier needs.
  for (int k = tid; k < min(n_mine, kItemCap); k += kThreads) {
    const Item it = decode_direct(item0 + k * item_step);
    int later = 0;
    for (int j = k + 1; j < n_mine && !later; ++j) later = decode_direct(item0 + j * item_step).active ? 1 : 0;
    ptx::sts128(item_tab + 32 * k, it.i0, it.h, it.b, it.len);
    ptx::sts128(item_tab + 32 * k + 16, it.rb, it.S, later, 0);
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  // k = position in this CTA's list; every loop below carries it along (no division by the grid size per decode)
  auto decode = [&](int item, int k) {
    if (k >= kItemCap) return decode_direct(item);
    Item it;
    const float4 a = lds_f32x4(item_tab + 32 * k), c = lds_f32x4(item_tab + 32 * k + 16);
    it.i0 = __float_as_int(a.x), it.h = __float_as_int(a.y), it.b = __float_as_int(a.z), it.len = __float_as_int(a.w);
    it.rb = __float_as_int(c.x), it.S = __float_as_int(c.y);
    finish(it);
    return it;
  };
  auto has_next_active = [&](int item, int k) {
    if (k < kItemCap) {
      uint32_t later;
      asm volatile("ld.shared.b32 %0, [%1];" : "=r"(later) : "r"(item_tab + 32 * k + 24) : "memory");
      return later != 0;
    }
    for (int j = item + item_step; j < p.n_items; j += item_step)
      if (decode_direct(j).active) return true;
    return false;
  };

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;" ::: "memory");
    if (warp == 0) {
      // ---------------------------------------------------------------------------------- TMA producer
      if (lane == 0) {
        int base_kv = 0, base_gb = 0;  // K/V tiles and band blocks loaded so far: ring positions stay continuous
        for (int item = item0, ik = 0; item < p.n_items; item += item_step, ++ik) {
          const Item w = decode(item, ik);
          if (!w.active) continue;
          const int r0 = T - 1 - w.i0 - (kBM - 1);  // band row of G column 0 of block 0 (may be < 0: TMA zero-fills)
          auto load_band_block = [&](int g) {
            if (g >= w.n_gb) return;
            const int idx = base_gb + g;
            const int slot = idx % kBandSlots, use = idx / kBandSlots;
            ptx::mbar_wait_a(band_empty + 8 * slot, (use & 1) ^ 1);
            ptx::mbar_arrive_expect_tx_a(band_full + 8 * slot, kBlockBytes);
            ptx::tma_load_2d_a(sbase + kOffBand + slot * kBlockBytes, &tmP, band_full + 8 * slot, w.h * kDK, r0 + 64 * g);
          };
          auto load_kv = [&](int kt) {
            const int idx = base_kv + kt;
            const int st = idx % kKVStages, use = idx / kKVStages;
            ptx::mbar_wait_a(kv_empty + 8 * st, (use & 1) ^ 1);
            ptx::mbar_arrive_expect_tx_a(kv_full + 8 * st, kKVBytes);
            const uint32_t dst = sbase + kOffKV + st * kKVBytes;
            ptx::tma_load_2d_a(dst, &tmKV, kv_full + 8 * st, 2 * p.Dp + w.h * kDK, w.rb + kt * kBN);
            ptx::tma_load_2d_a(dst + kKBytes, &tmKV, kv_full + 8 * st, 3 * p.Dp + w.h * kDK, w.rb + kt * kBN);
          };
          load_band_block(0);
          load_band_block(1);
          load_band_block(2);
          load_kv(0);
          load_band_block(3);
          for (int kt = 1; kt < w.n_kt; ++kt) {
            load_kv(kt);
            load_band_block(kt + 3);
          }
          base_kv += w.n_kt;
          base_gb += w.n_gb;
        }
      }
    } else if (warp == 1 || warp == 2) {
      // ---------------------------------------------------------------------------------- S / PV issuer of a set
      const int s = warp - 1;
      constexpr uint32_t idesc_s = ptx::make_idesc_bf16(kBM, kBN, 0, 0);
      constexpr uint32_t idesc_o = ptx::make_idesc_bf16(kBM, kDK, 0, 1);  // B = V is MN-major (keys x dk rows)
      const uint32_t tQu = tmem_base + kColQ;
      const uint32_t tS = tmem_base + kColS + s * 64;
      const uint32_t tP = tmem_base + kColP + s * 32;
      int base_kv = 0, base_it = 0, n_act = 0;
      for (int item = item0, ik = 0; item < p.n_items; item += item_step, ++ik) {
        const Item w = decode(item, ik);
        if (!w.active) continue;
        ptx::mbar_wait_a(qu_ready, n_act & 1);
        ptx::tc_fence_after();
        if (lane == 0) ptx::mbar_arrive_a(role_sync);
        int it = 0;
        for (int kt = s; kt < w.n_kt; kt += 2, ++it) {
          const int gi = base_it + it;
          const int idx = base_kv + kt;
          const int kvs = idx % kKVStages;
          const uint32_t st = sbase + kOffKV + kvs * kKVBytes;
          const uint64_t dK = ptx::make_sdesc_sw128(st, 16, 1024);
          const uint64_t dV = ptx::make_sdesc_sw128(st + kKBytes, 1024, 1024);
          ptx::mbar_wait_a(kv_full + 8 * kvs, (idx / kKVStages) & 1);
          ptx::mbar_wait_a(s_free + 8 * s, (gi & 1) ^ 1);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < kDK / 16; ++k) ptx::umma_bf16_ts(tS, tQu + 8 * k, dK + 2 * k, idesc_s, k != 0);
            ptx::tc_commit_a(sg_full + 8 * s);
          }
          __syncwarp();
          ptx::mbar_wait_a(p_ready + 8 * s, gi & 1);
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
        base_it += it;
        base_kv += w.n_kt;
        ++n_act;
      }
    } else {
      // ---------------------------------------------------------------------------------- G ring issuer
      constexpr uint32_t idesc_g = make_idesc_f16_f16acc(kBM, 64);
      const uint32_t tQv = tmem_base + kColQ + 32;
      const uint32_t band_base = sbase + kOffBand;
      int base_gb = 0, n_act = 0;
      // scalars, not arrays: an index that is only known at run time puts an array in LOCAL memory, and the loads showed
      // up as long-scoreboard stalls on the address arithmetic that follows (ncu source page)
      int base_it0 = 0, base_it1 = 0, prev_its0 = 0, prev_its1 = 0;
      for (int item = item0, ik = 0; item < p.n_items; item += item_step, ++ik) {
        const Item w = decode(item, ik);
        if (!w.active) continue;
        ptx::mbar_wait_a(qv_ready, n_act & 1);
        if (lane == 0) ptx::mbar_arrive_a(role_sync);
        // every window of the previous item has left the ring (the sets cannot be further: their next windows need
        // the blocks issued below)
        if (prev_its0 > 0) ptx::mbar_wait_a(g_free, (base_it0 - 1) & 1);
        if (prev_its1 > 0) ptx::mbar_wait_a(g_free + 8, (base_it1 - 1) & 1);
        for (int g = 0; g < w.n_gb; ++g) {
          const int idx = base_gb + g;
          const int bs = idx % kBandSlots;
          const uint64_t dB = ptx::make_sdesc_sw128(band_base + bs * kBlockBytes, 16, 1024);
          const uint32_t tG = tmem_base + kColG + (idx % kGSlots) * 64;
          ptx::mbar_wait_a(band_full + 8 * bs, (idx / kBandSlots) & 1);
          // ring slot idx % 4 held block g - 4 of this item, read by key tiles g-6, g-5, g-4.  Tile g-5 (the other
          // set's) was waited for at step g-1 and tile g-6 precedes g-4 in its set: one wait per step covers all three
          if (g >= 4 && g - 4 < w.n_kt) {
            const int s = (g - 4) & 1;
            ptx::mbar_wait_a(g_free + 8 * s, ((s ? base_it1 : base_it0) + ((g - 4) >> 1)) & 1);
          }
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < kDK / 16; ++k) ptx::umma_bf16_ts(tG, tQv + 8 * k, dB + 2 * k, idesc_g, k != 0);
            ptx::tc_commit_a(g_full + 8 * (idx % kGSlots));
            ptx::tc_commit_a(band_empty + 8 * bs);
          }
          __syncwarp();
        }
        base_gb += w.n_gb;
        prev_its0 = (w.n_kt + 1) / 2, prev_its1 = w.n_kt / 2;
        base_it0 += prev_its0, base_it1 += prev_its1;
        ++n_act;
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;" ::: "memory");
    // ---------------------------------------------------------------------------------- softmax warps
    const int quarter = warp & 3;
    const int set = (warp - 4) >> 2;
    const int ii = quarter * 32 + lane;  // query row inside the tile == TMEM lane
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    const uint32_t tS = t_lane + kColS + set * 64;
    const uint32_t tP = t_lane + kColP + set * 32;
    const int sh = 31 - lane;
    // 48 packed fp16 pairs per row, pitch 96 words plus a 16-byte skew: conflict-free 16-byte stores and 4-byte loads (attention_tc.cu)
    const uint32_t shift_row = sbase + kOffShift + (warp - 4) * kShiftBytes + lane * 96 * 4 +
                               static_cast<uint32_t>(((lane >> 1) + 4 * (lane & 1)) & 7) * 16;
    const int wcol = 96 - 32 * quarter;  // window start inside the concatenation of ring blocks kt, kt+1, kt+2
    const uint32_t xrow = sbase + kOffX + ii * kXPitch * 4;
    const float scale = p.scale_log2;

    // this thread's row of Q+u (set 0) / Q+v (set 1) of an item: 64 bf16
    uint32_t qw[32];
    auto fetch_q = [&](int item, int k) {
      const Item f = decode(item, k);
      const int h = f.h;
      const int i = f.i0 + ii;
      if (i < f.S) {
        const uint4* src = reinterpret_cast<const uint4*>(p.qkv + (static_cast<long long>(f.rb) + i) * (4 * p.Dp) +
                                                          set * p.Dp + h * kDK);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint4 u = __ldg(src + c);
          qw[4 * c] = u.x, qw[4 * c + 1] = u.y, qw[4 * c + 2] = u.z, qw[4 * c + 3] = u.w;
        }
      } else {
#pragma unroll
        for (int c = 0; c < 32; ++c) qw[c] = 0u;
      }
    };
    if (item0 < p.n_items) fetch_q(item0, 0);

    int base_gb = 0, n_act = 0;
    int base_mine = 0, base_other = 0;  // tiles this set / the other set has processed (scalars: see the G issuer)
    bool pre_stored = false;
    // qw -> the TMEM A operand of the item that `n_started` active items precede.  Every MMA of the item before it has
    // completed when this is called (both sets passed their last o_full wait and the exchange barrier; the last window
    // wait covered the last G block).  Parity waits tell the current phase from the previous one only: nobody may
    // signal item n before all three issuer warps have passed their operand wait of item n - 1 (an issuer with no tile
    // in an item could otherwise be lapped).
    auto store_q = [&](int n_started) {
      if (set == 1) {  // the G MMA takes fp16 operands: (q + v) / 16 as fp16
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&qw[c]));
          qw[c] = pack_f16x2(f.x * kGScaleInv, f.y * kGScaleInv);
        }
      }
      ptx::tmem_st_x32(t_lane + kColQ + set * 32, qw);
      ptx::tc_wait_st();
      ptx::tc_fence_before();
      if (n_started > 0) ptx::mbar_wait_a(role_sync, (n_started - 1) & 1);
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_a(set == 0 ? qu_ready : qv_ready);
    };
    for (int item = item0, ik = 0; item < p.n_items; item += item_step, ++ik) {
      const Item w = decode(item, ik);
      const int i = w.i0 + ii;
      if (!w.active) {
        if (set == 0 && i < w.S) {
          uint4* o = reinterpret_cast<uint4*>(p.ctx + (static_cast<long long>(w.rb) + i) * p.Dp + w.h * kDK);
#pragma unroll
          for (int c = 0; c < 8; ++c) o[c] = make_uint4(0, 0, 0, 0);
        }
        if (item + item_step < p.n_items) fetch_q(item + item_step, ik + 1);
        continue;
      }
      const int len = w.len, n_kt = w.n_kt;
      // ---- operand row -> TMEM, unless the tail of the previous item already did it (see below)
      if (!pre_stored) store_q(n_act);
      pre_stored = false;
      if (item + item_step < p.n_items) fetch_q(item + item_step, ik + 1);  // lands while this item's key tiles run

      auto fetch_window = [&](int kt) {
        const int last = base_gb + kt + 2;  // blocks complete in order
        ptx::mbar_wait_a(g_full + 8 * (last % kGSlots), (last / kGSlots) & 1);
        ptx::tc_fence_after();
        uint32_t wv[49];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int wc = wcol + 32 * c;
          const int blk = base_gb + kt + (wc >> 6);
          ptx::tmem_ld_x16_pack16(t_lane + kColG + (blk % kGSlots) * 64 + (wc & 63), &wv[16 * c]);
        }
        ptx::tc_wait_ld();
        wv[48] = 0u;
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_a(g_free + 8 * set);
        // odd shifts: move the row down by one half so that the halves (31 - lane) + 2 j, + 2 j + 1 share a word
        const uint32_t sel = (sh & 1) ? 0x5432u : 0x3210u;
#pragma unroll
        for (int m = 0; m < 48; ++m) wv[m] = prmt(wv[m], wv[m + 1], sel);
#pragma unroll
        for (int q = 0; q < 12; ++q) ptx::sts128(shift_row + q * 16, wv[4 * q], wv[4 * q + 1], wv[4 * q + 2], wv[4 * q + 3]);
      };

      float o_acc[kDK];
#pragma unroll
      for (int c = 0; c < kDK; ++c) o_acc[c] = 0.f;
      float m_run = -INFINITY, l_run = 0.f;

      if (set < n_kt) fetch_window(set);
      int it = 0;
      for (int kt = set; kt < n_kt; kt += 2, ++it) {
        const int j0 = kt * kBN;
        const int gi = base_mine + it;
        // the shifted window row was stored a whole P V MMA ago: read it while the S MMA of this tile is still in flight
        uint32_t gw[32];
        lds_u32x32(shift_row + (sh >> 1) * 4, gw);
        ptx::mbar_wait_a(sg_full + 8 * set, gi & 1);
        ptx::tc_fence_after();
        float sv[kBN];
        {
          uint32_t s0r[32], s1r[32];
          ptx::tmem_ld_x32(tS, s0r);
          ptx::tmem_ld_x32(tS + 32, s1r);
          ptx::tc_wait_ld();
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
        // the exponentials of consecutive key tiles take turns on the MUFU pipe (tile kt after tile kt-1)
        // (with one tile per set the order does not matter and set 1 need not idle through set 0's write-back of the
        // previous item: 128 x 100 frames x 4 heads 30.8 -> 29.5 us; with more tiles the strict order measures better)
        if (kt > (n_kt <= 2 ? 1 : 0)) ptx::mbar_wait_a(exp_done + 8 * (set ^ 1), (base_other + (set == 0 ? it - 1 : it)) & 1);
        float mx4[4] = {sv[0], sv[1], sv[2], sv[3]};
#pragma unroll
        for (int c = 4; c < kBN; ++c) mx4[c & 3] = fmaxf(mx4[c & 3], sv[c]);
        const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
        const float m_new = fmaxf(m_run, mx);  // finite: every tile holds at least one key j < len
        const float ms = m_new * scale;
        const float alpha = fast_exp2(fmaf(m_run, scale, -ms));
        float2 rs4[4] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
        uint32_t pw[32];
#pragma unroll
        for (int m = 0; m < 32; ++m) {  // scalar here (the packed forms of attention_tc.cu measure slower in this kernel), same order
          const float2 e = make_float2(fast_exp2(fmaf(sv[2 * m], scale, -ms)), fast_exp2(fmaf(sv[2 * m + 1], scale, -ms)));
          rs4[m & 3].x += e.x, rs4[m & 3].y += e.y;
          pw[m] = prmt(__float_as_uint(e.x) + 0x8000u, __float_as_uint(e.y) + 0x8000u, 0x7632u);
        }
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_a(exp_done + 8 * set);
        ptx::tmem_st_x32(tP, pw);
        const float rsum = ((rs4[0].x + rs4[1].x) + (rs4[2].x + rs4[3].x)) + ((rs4[0].y + rs4[1].y) + (rs4[2].y + rs4[3].y));
        l_run = fmaf(l_run, alpha, rsum);
        m_run = m_new;
        ptx::tc_wait_st();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_a(p_ready + 8 * set);
        if (kt + 2 < n_kt) fetch_window(kt + 2);  // the G window of this set's next tile, while the P V MMA runs
        ptx::mbar_wait_a(o_full + 8 * set, gi & 1);
        ptx::tc_fence_after();
        {
          uint32_t a0[32], a1[32];
          ptx::tmem_ld_x32(tS, a0);
          ptx::tmem_ld_x32(tS + 32, a1);
          ptx::tc_wait_ld();
#pragma unroll
          for (int c = 0; c < 32; ++c) {
            o_acc[c] = fmaf(o_acc[c], alpha, __uint_as_float(a0[c]));
            o_acc[32 + c] = fmaf(o_acc[32 + c], alpha, __uint_as_float(a1[c]));
          }
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_a(s_free + 8 * set);
      }
      base_gb += w.n_gb;
      base_mine += set == 0 ? (n_kt + 1) / 2 : n_kt / 2;
      base_other += set == 0 ? n_kt / 2 : (n_kt + 1) / 2;
      ++n_act;

      // ---- merge the two sets (log-sum-exp) through the exchange buffer and write the context rows.  Set 1 goes
      // straight on to the next item; it cannot reach its next exchange write before set 0 has read this one (the next
      // item's S MMAs wait for set 0's operand row).
      if (set == 1) {
        // set 0 has read the previous item's exchange rows (it arrives on barrier 2 after its reads)
        if (n_act > 1) asm volatile("bar.sync 2, 256;" ::: "memory");
        ptx::sts128(xrow, __float_as_uint(m_run), __float_as_uint(l_run), 0u, 0u);
#pragma unroll
        for (int c = 0; c < kDK / 4; ++c)
          ptx::sts128(xrow + 16 + 16 * c, __float_as_uint(o_acc[4 * c]), __float_as_uint(o_acc[4 * c + 1]),
                      __float_as_uint(o_acc[4 * c + 2]), __float_as_uint(o_acc[4 * c + 3]));
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      // The next item's operand goes into TMEM BEFORE this item's merge and write-back: its S and G MMAs then run while
      // set 0 is still busy with the context rows (qw holds the next item's row since the top of this iteration).
      if (item + item_step < p.n_items && decode(item + item_step, ik + 1).active) {
        store_q(n_act);
        pre_stored = true;
      }
      if (set == 0) {
        const float4 ml = lds_f32x4(xrow);
        const float m1 = ml.x, l1 = ml.y;
        const float m = fmaxf(m_run, m1);  // set 0 always owns key tile 0, so m is finite
        const float w0 = fast_exp2((m_run - m) * scale), w1 = fast_exp2((m1 - m) * scale);
        const float l = l_run * w0 + l1 * w1;
        const float inv = (i < len && l > 0.f) ? 1.f / l : 0.f;  // padded query rows -> zeros
        const float c0 = w0 * inv, c1 = w1 * inv;
        if (i < w.S) {
          uint4* o = reinterpret_cast<uint4*>(p.ctx + (static_cast<long long>(w.rb) + i) * p.Dp + w.h * kDK);
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
        // the exchange rows are free again; set 1 waits for this before its next write (not after the last item)
        if (has_next_active(item, ik)) asm volatile("bar.arrive 2, 256;" ::: "memory");
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

int launch_attn_tcp(const AttnDesc& a, cudaStream_t st, std::string* err) {
  if ((a.tiles == nullptr && a.B <= 0) || a.T <= 0) return 0;
  if (a.dkp != kDK) {
    if (err) *err = "attn_tcp: padded head dim must be 64";
    return -1;
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
  {
    // fp16 copy of the projections the G MMA reads (converted in place once per forward by the engine; see attention_tc.cu)
    const void* pos16 = attn_pos_f16(a, Dp, st);
    uint64_t dims[2] = {static_cast<uint64_t>(Dp), static_cast<uint64_t>(2 * a.T - 1)};
    uint64_t strides[1] = {static_cast<uint64_t>(a.pos_f16 ? a.ld_pos : Dp) * 2};
    uint32_t box[2] = {kDK, 64};
    if (!encode_tmap_bf16(&tmP, pos16, 2, dims, strides, box, err)) return -1;
  }
  static bool configured[64] = {};
  static int sms[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(rel_attn_tcp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTotal);
    if (e != cudaSuccess) {
      if (err) *err = std::string("cudaFuncSetAttribute(attn_tcp): ") + cudaGetErrorString(e);
      return static_cast<int>(e);
    }
    cudaDeviceGetAttribute(&sms[dev & 63], cudaDevAttrMultiProcessorCount, dev);
    if (sms[dev & 63] <= 0) sms[dev & 63] = 148;
    configured[dev & 63] = true;
  }
  AttnPParams p;
  p.qkv = reinterpret_cast<const bf16*>(a.qkv);
  p.lens = a.lens;
  p.ctx = reinterpret_cast<bf16*>(a.ctx);
  p.T = a.T;
  p.Dp = Dp;
  p.H = a.H;
  p.n_qt = a.tiles != nullptr ? a.n_tiles : (a.T + kBM - 1) / kBM;
  p.n_items = (a.tiles != nullptr ? 1 : a.B) * a.H * p.n_qt;
  p.tiles = a.tiles;
  p.scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(a.dk));
  const int grid = p.n_items < sms[dev & 63] ? p.n_items : sms[dev & 63];
  cudaError_t e = launch_pdl(rel_attn_tcp_kernel, dim3(grid), dim3(kThreads), kSmemTotal, st, tmKV, tmP, p);
  if (e != cudaSuccess) {
    if (err) *err = std::string("attn_tcp launch: ") + cudaGetErrorString(e);
    return static_cast<int>(e);
  }
  return 0;
}

}  // namespace cfb
