// Transducer greedy decode on the encoder output (SURVEY.md 8(f) rank 4): the prediction network (Embedding + one LSTM
// layer, modules/rnnt.py:190-283), the joint network (modules/rnnt.py:951-1008) and the greedy_batch loop
// (parts/submodules/rnnt_greedy_decoding.py:454-616) as ONE persistent cooperative kernel.
//
// The reference runs ~15 small PyTorch kernels plus a host synchronisation (`blank_mask.all()`) per symbol step.  Here
//   * joint.enc is applied to every frame up front by the tcgen05 GEMM (bf16 hi/lo split operands, fp32 accumulation:
//     A' = [hi | hi | lo], W' = [hi | lo | hi], so the product keeps fp32-level accuracy),
//   * one CTA per SM keeps ITS rows of the LSTM, joint.pred and joint_net weights in shared memory in fp32 for the whole
//     decode (weight-stationary: 17.4 MB / 148 SMs = 133 KB per SM for the Conformer-Transducer sizes), so a step moves
//     only activations (a few KB per utterance) through L2,
//   * utterances advance in lock-step "iterations": every active utterance evaluates the joint at its own frame; the ones
//     that emitted a symbol then run the LSTM cell and joint.pred.  An utterance that produced a blank keeps its
//     prediction-network output (the reference recomputes the identical value), so the LSTM runs once per emitted symbol,
//   * the per-utterance control state (frame, symbols at this frame, last label, ...) is replicated in every CTA and
//     advanced deterministically from the one exchanged datum: the arg-max, combined across CTAs with a packed 64-bit
//     atomicMax (value bits | inverted index => first index wins ties like torch.max),
//   * phases are separated by a grid barrier (1 per blank-only iteration, 3 when something was emitted).
#include <float.h>
#include <stdlib.h>

#include "../../include/cfb.h"
#include "common.cuh"
#include "rnnt_common.cuh"

namespace cfb {
namespace {

constexpr int kThreads = 512;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxB = 128;  // utterances per launch (control state lives in shared memory)
constexpr int kMaxTile = 32;  // utterances staged in shared memory at a time (the staging buffer takes what the weights leave)
constexpr int kJointRound = 1;  // (e0, e1, q) float4 triples per thread and joint staging round
constexpr int kStageRound = 2;  // float4 per thread and LSTM / pred staging round
constexpr int kHardSymbolLimit = 4096;  // symbols per frame when max_symbols is unlimited (flag bit 1 if ever reached)

struct RnntParams {
  // sizes
  int E, H, J, V1, act, B, T, max_symbols, max_tokens;
  // weights (fp32, reference state_dict layout)
  const float *embed, *w_ih, *w_hh, *b_ih, *b_hh, *w_pred, *b_pred, *w_out, *b_out;
  // activations
  const float* encp;  // (B*T, J) = joint.enc(encoded)
  const int32_t* lens;
  float* hbuf;   // [2][B][H]
  float* predp;  // [B][J]
  unsigned long long* slots;  // [3][2][kMaxB]
  unsigned int* counter;      // grid barrier
  // outputs
  int32_t *tokens, *timesteps, *n_tokens, *flags;
  float *scores, *h_out, *c_out;
  int umax, pmax, jmax;  // rows per CTA (ceil)
  int stage_floats;      // size of the activation staging buffer
};

// NI > 0: K4 == 32 * NI, fully unrolled (the shared-memory loads of an iteration are issued ahead of the FMAs of the previous one).
template <int NI>
__device__ __forceinline__ void tile_dot_body(const float4* __restrict__ w, const float4* __restrict__ w1, const float4* __restrict__ w2,
                                              const float4* __restrict__ w3, const float4* __restrict__ z0,
                                              const float4* __restrict__ z1, int K4, int lane, float acc[4][2]) {
  auto step = [&](int k4) {
    const float4 a0 = z0[k4], a1 = z1[k4];
    const float4 v0 = w[k4], v1 = w1[k4], v2 = w2[k4], v3 = w3[k4];
    acc[0][0] = dot4(v0, a0, acc[0][0]), acc[0][1] = dot4(v0, a1, acc[0][1]);
    acc[1][0] = dot4(v1, a0, acc[1][0]), acc[1][1] = dot4(v1, a1, acc[1][1]);
    acc[2][0] = dot4(v2, a0, acc[2][0]), acc[2][1] = dot4(v2, a1, acc[2][1]);
    acc[3][0] = dot4(v3, a0, acc[3][0]), acc[3][1] = dot4(v3, a1, acc[3][1]);
  };
  if (NI > 0) {
#pragma unroll
    for (int i = 0; i < NI; ++i) step(lane + 32 * i);
  } else {
#pragma unroll 2
    for (int k4 = lane; k4 < K4; k4 += 32) step(k4);
  }
}
__device__ __forceinline__ void tile_dot(const float4* __restrict__ w, int row_stride4, int nrows, const float4* __restrict__ z0,
                                         const float4* __restrict__ z1, int K4, int lane, float acc[4][2]) {
  const float4* w1 = w + (nrows > 1 ? 1 : 0) * row_stride4;
  const float4* w2 = w + (nrows > 2 ? 2 : 0) * row_stride4;
  const float4* w3 = w + (nrows > 3 ? 3 : 0) * row_stride4;
  if (K4 == 160) tile_dot_body<5>(w, w1, w2, w3, z0, z1, K4, lane, acc);         // 640 (the transducer recipes' hidden sizes)
  else if (K4 == 320) tile_dot_body<10>(w, w1, w2, w3, z0, z1, K4, lane, acc);   // 1280 = [x | h]
  else tile_dot_body<0>(w, w1, w2, w3, z0, z1, K4, lane, acc);
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    acc[r][0] = warp_sum(acc[r][0]);
    acc[r][1] = warp_sum(acc[r][1]);
  }
}

// R (4 or 8) weight rows x 4 staged activation vectors: acc[r * 4 + s] += sum_k w[r][k] * z_s[k] over this lane's k, then a
// transposing butterfly (R * 4 - 1 shuffles instead of R * 20) leaves the warp total of accumulator i in lane i (and in
// lane i + 16 when R == 4): lane = row * 4 + vector.
template <int R, int NI>
__device__ __forceinline__ float tile_dot_r4(const float4* __restrict__ w, int row_stride4, int nrows, const float4* __restrict__ z,
                                             int z_stride4, const int zi[4], int K4, int lane) {
  constexpr int NV = R * 4;
  float acc[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) acc[i] = 0.f;
  auto step = [&](int k4) {
    float4 a[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) a[s] = z[zi[s] * z_stride4 + k4];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const float4 v = w[(r < nrows ? r : 0) * row_stride4 + k4];
#pragma unroll
      for (int s = 0; s < 4; ++s) acc[r * 4 + s] = dot4(v, a[s], acc[r * 4 + s]);
    }
  };
  if (NI > 0) {
#pragma unroll
    for (int i = 0; i < NI; ++i) step(lane + 32 * i);
  } else if (NI < 0) {  // -NI unrolled iterations, the last one partial (K4 not a multiple of 32)
#pragma unroll
    for (int i = 0; i < -NI; ++i)
      if (lane + 32 * i < K4) step(lane + 32 * i);
  } else {
    for (int k4 = lane; k4 < K4; k4 += 32) step(k4);
  }
#pragma unroll
  for (int half = NV / 2; half > 0; half >>= 1) {
    const bool up = (lane & half) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float send = up ? acc[i] : acc[i + half];
      const float keep = up ? acc[i + half] : acc[i];
      acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
    }
  }
#pragma unroll
  for (int o = NV; o < 32; o <<= 1) acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], o);
  return acc[0];
}

// compact list of the indices b < B with flag[b] != 0, in ascending order (identical in every CTA); returns the count
__device__ int build_list(const int* flag, int B, int* list, int* s_tmp) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const bool f = tid < B && flag[tid] != 0;
  const unsigned int m = __ballot_sync(0xffffffffu, f);
  if (lane == 0) s_tmp[w] = __popc(m);
  __syncthreads();
  int base = 0, total = 0;
  for (int i = 0; i < kWarps; ++i) {
    const int cnt = s_tmp[i];
    if (i < w) base += cnt;
    total += cnt;
  }
  if (f) list[base + __popc(m & ((1u << lane) - 1u))] = tid;
  __syncthreads();
  return total;
}

// Per-utterance control of a launch, replicated in every CTA and advanced identically from the one exchanged datum (the
// combined arg-max keys in p.slots): frame, symbols emitted at it, last label, which half of hbuf / s_c holds the pending
// prediction-network state, tokens emitted, length, score (CTA 0's copy is written out), active and emitted flags and
// their ascending lists.  Both greedy kernels run exactly this decode rule.
struct GreedyControl {
  double score[kMaxB];
  int t[kMaxB], sym[kMaxB], last[kMaxB], par[kMaxB], ntok[kMaxB], len[kMaxB];
  int active[kMaxB], emit[kMaxB], alist[kMaxB], elist[kMaxB];
  int tmp[kWarps];

  // Every utterance starts at frame 0 with the SOS step pending (joint.pred of its first prediction-network output).
  __device__ void init(const RnntParams& p) {
    const int tid = threadIdx.x;
    if (tid < kMaxB) {
      const int n = tid < p.B ? min(max(p.lens[tid], 0), p.T) : 0;
      len[tid] = n;
      t[tid] = 0;
      sym[tid] = 0;
      last[tid] = p.V1 - 1;
      par[tid] = 0;
      ntok[tid] = 0;
      score[tid] = 0.0;
      active[tid] = n > 0;
      emit[tid] = tid < p.B;
    }
    __syncthreads();
  }

  __device__ void build_lists(int B, int* n_emit, int* n_active) {
    *n_emit = build_list(emit, B, elist, tmp);
    *n_active = build_list(active, B, alist, tmp);
  }

  // Consumes the keys of lock-step iteration `it` (frame t and, only after a blank, the speculatively evaluated t + 1),
  // appends the emitted token (CTA 0), clears the slots of iteration it + 2 (the three sets rotate: every CTA finished
  // reading them in iteration it - 1) and rebuilds the lists.
  __device__ void update(const RnntParams& p, unsigned int it, int* n_emit, int* n_active) {
    const int tid = threadIdx.x, cta = blockIdx.x, blank = p.V1 - 1;
    if (tid < kMaxB) {
      int e = 0;
      if (tid < p.B && active[tid]) {
        int tt = t[tid], sy = sym[tid];
        const int n_len = len[tid];
        for (int f = 0; f < 2; ++f) {
          float v;
          int k;
          unpack_key(__ldcg(&p.slots[((it % 3) * 2 + f) * kMaxB + tid]), &v, &k);
          if (k == blank) {
            ++tt;
            sy = 0;
            if (tt >= n_len) break;
            continue;
          }
          e = 1;
          const int n = ntok[tid];
          if (cta == 0) {
            if (n < p.max_tokens) {
              p.tokens[static_cast<size_t>(tid) * p.max_tokens + n] = k;
              p.timesteps[static_cast<size_t>(tid) * p.max_tokens + n] = tt;
            } else {
              atomicOr(p.flags, 1);
            }
            score[tid] += static_cast<double>(v);
          }
          ntok[tid] = n + 1;
          last[tid] = k;
          if (++sy >= (p.max_symbols > 0 ? p.max_symbols : kHardSymbolLimit)) {
            if (p.max_symbols <= 0 && cta == 0) atomicOr(p.flags, 2);  // runaway emission: the reference would not return
            ++tt;
            sy = 0;
          }
          break;  // the prediction network must advance before the next joint evaluation
        }
        t[tid] = tt;
        sym[tid] = sy;
        active[tid] = tt < n_len;
      }
      emit[tid] = e;
      if (cta == 0) {
        p.slots[(((it + 2) % 3) * 2 + 0) * kMaxB + tid] = 0ull;
        p.slots[(((it + 2) % 3) * 2 + 1) * kMaxB + tid] = 0ull;
      }
    }
    __syncthreads();
    build_lists(p.B, n_emit, n_active);
  }

  // Results: the committed state is the half the pending one does not occupy.  This CTA's cell states are those of units
  // [u0, u0 + nu) in s_c [2][B][cstride].
  __device__ void write_results(const RnntParams& p, const float* s_c, int cstride, int u0, int nu) {
    const int tid = threadIdx.x, cta = blockIdx.x, B = p.B, H = p.H;
    for (int i = tid; i < nu * B; i += kThreads) {
      const int u = i % nu, b = i / nu;
      p.c_out[static_cast<size_t>(b) * H + u0 + u] = s_c[((par[b] ^ 1) * B + b) * cstride + u];
    }
    for (int i = cta * kThreads + tid; i < B * H; i += gridDim.x * kThreads) {
      const int b = i / H, u = i % H;
      p.h_out[i] = __ldcg(p.hbuf + (static_cast<size_t>(par[b] ^ 1) * B + b) * H + u);
    }
    if (cta == 0 && tid < B) {
      p.n_tokens[tid] = ntok[tid];
      p.scores[tid] = static_cast<float>(score[tid]);
    }
  }
};

__global__ void __launch_bounds__(kThreads, 1) rnnt_greedy_kernel(const RnntParams p) {
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = gridDim.x, cta = blockIdx.x;
  const int H = p.H, J = p.J, V1 = p.V1, B = p.B, K2 = 2 * p.H;

  int u_lo, u_hi, p_lo, p_hi, j_lo, j_hi;
  row_range(H, cta, G, &u_lo, &u_hi);
  row_range(J, cta, G, &p_lo, &p_hi);
  row_range(V1, cta, G, &j_lo, &j_hi);
  const int nu = u_hi - u_lo, np = p_hi - p_lo, nj = j_hi - j_lo;

  // ---- shared memory carve-up ------------------------------------------------------------------------------------
  float* s_wl = smem;                                   // [umax][4][2H]  LSTM rows of my units: [w_ih row | w_hh row]
  float* s_wp = s_wl + static_cast<size_t>(p.umax) * 4 * K2;  // [pmax][H]
  float* s_wj = s_wp + static_cast<size_t>(p.pmax) * H;       // [jmax][J]
  float* s_bl = s_wj + static_cast<size_t>(p.jmax) * J;       // [umax][4] b_ih + b_hh
  float* s_c = s_bl + p.umax * 4;                             // [2][B][umax] cell state of my units
  float4* s_stage = reinterpret_cast<float4*>(s_c + ((static_cast<size_t>(2) * B * p.umax + 3) / 4) * 4);  // p.stage_floats
  const int J4 = J / 4, H4 = H / 4, K24 = K2 / 4;
  __shared__ unsigned long long s_best[2 * kMaxB];  // [frame 0 | frame 1][utterance]
  __shared__ GreedyControl ctl;

  load_row_weights(p, u_lo, nu, p_lo, np, j_lo, nj, s_wl, s_bl, s_wp, s_wj);
  ctl.init(p);

  // ---- SOS: pending = LSTM(x = 0, h = 0, c = 0) = f(bias) for every utterance; committed state = 0 (hbuf[1] is zeroed) --
  for (int i = tid; i < nu * B; i += kThreads) {
    const int ul = i % nu, b = i / nu;
    const float* bl = s_bl + ul * 4;
    const float c1 = sigmoidf_(bl[0]) * tanhf(bl[2]);  // f * 0 + i * g
    const float h1 = sigmoidf_(bl[3]) * tanhf(c1);
    s_c[(0 * B + b) * p.umax + ul] = c1;
    s_c[(1 * B + b) * p.umax + ul] = 0.f;
    p.hbuf[(static_cast<size_t>(0) * B + b) * H + u_lo + ul] = h1;
  }
  unsigned int bar_target = 0;
  int n_emit, n_active;
  ctl.build_lists(B, &n_emit, &n_active);
  grid_sync(p.counter, bar_target);

  bool first = true;
  for (unsigned int it = 0;; ++it) {
    if (!first) {
      // ---- joint: logits of my rows for every active utterance at its frame, arg-max ----------------------------------
      // Two frames per utterance are evaluated with the same prediction-network output: if the first is blank (the common
      // case) the second is already the answer for the next frame, so a lock-step iteration consumes up to two frames.
      if (tid < 2 * kMaxB) s_best[tid] = 0ull;
      __syncthreads();
      const int nchunks = (nj + 7) >> 3;
      // utterances staged at a time (the tile sizes are recomputed in each phase rather than kept live across the loop):
      // the joint tasks take groups of 4 staged vectors, two per utterance; the LSTM / pred tasks take pairs
      const int tile_s = (min(kMaxTile, p.stage_floats / J) & ~3) >> 1;
      for (int s0 = 0; nj > 0 && s0 < n_active; s0 += tile_s) {
        const int ns = min(tile_s, n_active - s0), total = ns * J4;
        // stage z_f = act(enc_proj[b, t_b + f] + pred_proj[b]), f = 0, 1: all loads of a round are issued before the first use
        for (int base = 0; base < total; base += kThreads * kJointRound) {
          float4 e0[kJointRound], e1[kJointRound], q[kJointRound];
#pragma unroll
          for (int u = 0; u < kJointRound; ++u) {
            const int idx = base + u * kThreads + tid;
            if (idx < total) {
              const int bb = ctl.alist[s0 + idx / J4], k4 = idx % J4, t0 = ctl.t[bb], t1 = min(t0 + 1, ctl.len[bb] - 1);
              e0[u] = __ldg(reinterpret_cast<const float4*>(p.encp + (static_cast<size_t>(bb) * p.T + t0) * J) + k4);
              e1[u] = __ldg(reinterpret_cast<const float4*>(p.encp + (static_cast<size_t>(bb) * p.T + t1) * J) + k4);
              q[u] = ldcg4(p.predp + static_cast<size_t>(bb) * J + k4 * 4);
            }
          }
#pragma unroll
          for (int u = 0; u < kJointRound; ++u) {
            const int idx = base + u * kThreads + tid;
            if (idx < total) {
              const int i = idx / J4, k4 = idx % J4;
              float4 z;
              z.x = act_fn(e0[u].x + q[u].x, p.act), z.y = act_fn(e0[u].y + q[u].y, p.act);
              z.z = act_fn(e0[u].z + q[u].z, p.act), z.w = act_fn(e0[u].w + q[u].w, p.act);
              s_stage[(2 * i) * J4 + k4] = z;
              z.x = act_fn(e1[u].x + q[u].x, p.act), z.y = act_fn(e1[u].y + q[u].y, p.act);
              z.z = act_fn(e1[u].z + q[u].z, p.act), z.w = act_fn(e1[u].w + q[u].w, p.act);
              s_stage[(2 * i + 1) * J4 + k4] = z;
            }
          }
        }
        __syncthreads();
        const int nv = 2 * ns, ngroups = (nv + 3) >> 2;  // staged vector v = 2 * utterance + frame
        for (int task = warp; task < ngroups * nchunks; task += kWarps) {
          const int grp = task % ngroups, ch = task / ngroups, r0 = ch * 8;
          int zi[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) zi[u] = min(4 * grp + u, nv - 1);
          const float4* wr = reinterpret_cast<const float4*>(s_wj) + r0 * J4;
          const float total = J4 == 160 ? tile_dot_r4<8, 5>(wr, J4, nj - r0, s_stage, J4, zi, J4, lane)
                                        : tile_dot_r4<8, 0>(wr, J4, nj - r0, s_stage, J4, zi, J4, lane);
          // lane = row * 4 + vector: bias, key, then the maximum over the 8 rows (lane bits 2..4)
          const int r = lane >> 2, v = 4 * grp + (lane & 3);
          unsigned long long key = 0ull;
          if (r0 + r < nj) key = pack_key(total + __ldg(p.b_out + j_lo + r0 + r), j_lo + r0 + r);
#pragma unroll
          for (int o = 4; o < 32; o <<= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
            key = other > key ? other : key;
          }
          if (lane < 4 && v < nv) atomicMax(&s_best[(v & 1) * kMaxB + ctl.alist[s0 + (v >> 1)]], key);
        }
        __syncthreads();
      }
      __syncthreads();
      if (nj > 0 && tid < 2 * n_active) {
        const int b = ctl.alist[tid >> 1], f = tid & 1;
        atomicMax(&p.slots[((it % 3) * 2 + f) * kMaxB + b], s_best[f * kMaxB + b]);
      }
      grid_sync(p.counter, bar_target);

      // ---- control update (replicated in every CTA) ---------------------------------------------------------------------
      ctl.update(p, it, &n_emit, &n_active);

      // ---- LSTM cell for the utterances that emitted: commit the pending state, compute the next one -----------------------
      if (n_emit > 0) {
        const int tile_l = min(kMaxTile, p.stage_floats / K2) & ~1;
        for (int s0 = 0; nu > 0 && s0 < n_emit; s0 += tile_l) {
          const int ns = min(tile_l, n_emit - s0), total = ns * K24;
          // stage [embed(last label) | h] of the utterances of this tile
          for (int base = 0; base < total; base += kThreads * kStageRound) {
            float4 v[kStageRound];
#pragma unroll
            for (int u = 0; u < kStageRound; ++u) {
              const int idx = base + u * kThreads + tid;
              if (idx < total) {
                const int bb = ctl.elist[s0 + idx / K24], k4 = idx % K24;
                v[u] = k4 < H4 ? __ldg(reinterpret_cast<const float4*>(p.embed + static_cast<size_t>(ctl.last[bb]) * H) + k4)
                               : ldcg4(p.hbuf + (static_cast<size_t>(ctl.par[bb]) * B + bb) * H + (k4 - H4) * 4);
              }
            }
#pragma unroll
            for (int u = 0; u < kStageRound; ++u) {
              const int idx = base + u * kThreads + tid;
              if (idx < total) s_stage[idx] = v[u];
            }
          }
          __syncthreads();
          const int ngr = (ns + 3) >> 2;  // tasks = (hidden unit: its 4 gate rows) x (group of 4 utterances)
          for (int task = warp; task < ngr * nu; task += kWarps) {
            const int grp = task % ngr, ul = task / ngr;
            int zi[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) zi[u] = min(4 * grp + u, ns - 1);
            const float4* wr = reinterpret_cast<const float4*>(s_wl) + static_cast<size_t>(ul) * 4 * K24;
            const float total = K24 == 320 ? tile_dot_r4<4, 10>(wr, K24, 4, s_stage, K24, zi, K24, lane)
                                           : tile_dot_r4<4, 0>(wr, K24, 4, s_stage, K24, zi, K24, lane);
            // lane = gate * 4 + utterance: hand the four gate pre-activations of utterance u to lane u
            const int u = lane & 3;
            const float* bl = s_bl + ul * 4;
            const float gi = __shfl_sync(0xffffffffu, total, u) + bl[0], gf = __shfl_sync(0xffffffffu, total, 4 + u) + bl[1];
            const float gg = __shfl_sync(0xffffffffu, total, 8 + u) + bl[2], go = __shfl_sync(0xffffffffu, total, 12 + u) + bl[3];
            if (lane < 4 && 4 * grp + u < ns) {
              const int b = ctl.elist[s0 + 4 * grp + u];
              const int par = ctl.par[b];
              const float c_old = s_c[(par * B + b) * p.umax + ul];
              const float c_new = sigmoidf_(gf) * c_old + sigmoidf_(gi) * tanhf(gg);
              const float h_new = sigmoidf_(go) * tanhf(c_new);
              s_c[((par ^ 1) * B + b) * p.umax + ul] = c_new;
              p.hbuf[(static_cast<size_t>(par ^ 1) * B + b) * H + u_lo + ul] = h_new;
            }
          }
          __syncthreads();
        }
        __syncthreads();
        if (tid < n_emit) ctl.par[ctl.elist[tid]] ^= 1;
        grid_sync(p.counter, bar_target);
      }
      if (n_active == 0) break;
    }
    first = false;

    // ---- joint.pred of the new prediction-network outputs -------------------------------------------------------------------
    if (n_emit > 0) {
      const int nchunks = (np + 3) >> 2;
      const int tile_p = min(kMaxTile, p.stage_floats / H) & ~1;
      for (int s0 = 0; np > 0 && s0 < n_emit; s0 += tile_p) {
        const int ns = min(tile_p, n_emit - s0), total = ns * H4;
        for (int base = 0; base < total; base += kThreads * kStageRound) {
          float4 v[kStageRound];
#pragma unroll
          for (int u = 0; u < kStageRound; ++u) {
            const int idx = base + u * kThreads + tid;
            if (idx < total) {
              const int bb = ctl.elist[s0 + idx / H4];
              v[u] = ldcg4(p.hbuf + (static_cast<size_t>(ctl.par[bb]) * B + bb) * H + (idx % H4) * 4);
            }
          }
#pragma unroll
          for (int u = 0; u < kStageRound; ++u) {
            const int idx = base + u * kThreads + tid;
            if (idx < total) s_stage[idx] = v[u];
          }
        }
        __syncthreads();
        const int npe = (ns + 1) >> 1;
        for (int task = warp; task < npe * nchunks; task += kWarps) {
          const int pr = task % npe, ch = task / npe, r0 = ch * 4;
          const int i0 = 2 * pr, i1 = (2 * pr + 1 < ns) ? 2 * pr + 1 : i0;
          float acc[4][2] = {};
          tile_dot(reinterpret_cast<const float4*>(s_wp) + r0 * H4, H4, np - r0, s_stage + i0 * H4, s_stage + i1 * H4, H4, lane, acc);
          const int b0 = ctl.elist[s0 + i0], b1 = ctl.elist[s0 + i1];
#pragma unroll
          for (int r = 0; r < 4; ++r) {
            if (r0 + r < np) {
              const int row = p_lo + r0 + r;
              const float bias = __ldg(p.b_pred + row);
              if (lane == 0) p.predp[static_cast<size_t>(b0) * J + row] = acc[r][0] + bias;
              if (lane == 1 && i1 != i0) p.predp[static_cast<size_t>(b1) * J + row] = acc[r][1] + bias;
            }
          }
        }
        __syncthreads();
      }
      grid_sync(p.counter, bar_target);
    }
    if (n_active == 0) break;
  }

  ctl.write_results(p, s_c, p.umax, u_lo, nu);
}

// ======================================================================================================================
// Cluster variant: the same decode with the weights split over rows ACROSS clusters of 4 CTAs and over K INSIDE a cluster.
// Cluster q owns a block of hidden units / joint.pred rows / output rows; rank r of the cluster keeps the K-quarter r of all
// of them, so a CTA stages only a quarter of every activation vector (the per-SM ingest from L2 was the limit of the
// row-only partition: every CTA read every utterance's vectors).  The four partial dot products of a row meet in the shared
// memory of the row's owner rank (st.shared::cluster) and are added there in rank order 0..3 -- a fixed order, so results
// do not depend on the batch or on timing.  One cluster barrier per tile; partial buffers are double-buffered, which is
// enough because a rank cannot pass barrier n + 1 before every rank has finished reading the partials of barrier n.
constexpr int kC = 4;            // CTAs per cluster
constexpr int kTileL = 16;       // utterances per LSTM tile
constexpr int kTileP = 32;       // utterances per joint.pred tile
constexpr int kTileV = 64;       // staged vectors per joint tile (32 utterances x 2 frames)

__device__ __forceinline__ uint32_t smem_addr_u32(const void* ptr) { return static_cast<uint32_t>(__cvta_generic_to_shared(ptr)); }
__device__ __forceinline__ void st_cluster_f32(const float* local_ptr, int rank, float v) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_addr_u32(local_ptr)), "r"(rank));
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(remote), "f"(v) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// owner rank of element i when n elements are split with row_range over kC ranks, and its index inside the owner's slice
__device__ __forceinline__ void owner_of(int i, int n, int* rank, int* local) {
  int o = 0, lo = 0;
#pragma unroll
  for (int c = 0; c < kC; ++c) {
    const int l = n * c / kC, h = n * (c + 1) / kC;
    if (i >= l && i < h) {
      o = c;
      lo = l;
    }
  }
  *rank = o;
  *local = i - lo;
}

__global__ void __launch_bounds__(kThreads, 1) rnnt_greedy_c4_kernel(const RnntParams p) {
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = gridDim.x, cta = blockIdx.x, NQ = G / kC, q = cta / kC, r = cta % kC;
  const int H = p.H, J = p.J, V1 = p.V1, B = p.B;
  const int Lq = H / 2, Hq = H / 4, Jq = J / 4;          // K slices (floats): LSTM [x | h], joint.pred, output layer
  const int Lq4 = Lq / 4, Hq4 = Hq / 4, Jq4 = Jq / 4;

  int uq_lo, uq_hi, pq_lo, pq_hi, jq_lo, jq_hi;          // the cluster's rows
  row_range(H, q, NQ, &uq_lo, &uq_hi);
  row_range(J, q, NQ, &pq_lo, &pq_hi);
  row_range(V1, q, NQ, &jq_lo, &jq_hi);
  const int nuq = uq_hi - uq_lo, npq = pq_hi - pq_lo, njq = jq_hi - jq_lo;
  int mu_lo, mu_hi, mp_lo, mp_hi;                        // the rows this rank finalises (relative to the cluster's)
  row_range(nuq, r, kC, &mu_lo, &mu_hi);
  row_range(npq, r, kC, &mp_lo, &mp_hi);
  const int nmu = mu_hi - mu_lo, nmp = mp_hi - mp_lo;
  const int nchunks = (njq + 7) >> 3;                    // output rows in chunks of 8; chunk c is finalised by rank c (host: <= kC)
  const int mumax = (p.umax + kC - 1) / kC, mpmax = (p.pmax + kC - 1) / kC;

  float* s_wl = smem;                                               // [umax][4][Lq]
  float* s_wp = s_wl + static_cast<size_t>(p.umax) * 4 * Lq;        // [pmax][Hq]
  float* s_wj = s_wp + static_cast<size_t>(p.pmax) * Hq;            // [jmax][Jq]
  float* s_bl = s_wj + static_cast<size_t>(p.jmax) * Jq;            // [mumax][4]
  float* s_c = s_bl + mumax * 4;                                    // [2][B][mumax]
  float* s_pj = s_c + ((static_cast<size_t>(2) * B * mumax + 3) / 4) * 4;  // [2][kC][8][kTileV]   partial logits
  float* s_pl = s_pj + 2 * kC * 8 * kTileV;                         // [2][kC][mumax][4][kTileL] partial gates
  float* s_pp = s_pl + 2 * kC * mumax * 4 * kTileL;                 // [2][kC][mpmax][kTileP]    partial joint.pred
  float4* s_stage = reinterpret_cast<float4*>(s_pp + ((2 * kC * mpmax * kTileP + 3) / 4) * 4);
  const int tile_s = min(kTileV / 2, p.stage_floats / (2 * Jq)) & ~1;   // utterances per joint tile (two vectors each)
  const int tile_l = min(kTileL, p.stage_floats / Lq) & ~3, tile_p = min(kTileP, p.stage_floats / Hq) & ~3;
  __shared__ unsigned long long s_best[2 * kMaxB];
  __shared__ GreedyControl ctl;

  // ---- my K-quarter of the cluster's weight rows (once) --------------------------------------------------------------------
  for (int i = tid; i < nuq * 4 * Lq4; i += kThreads) {
    const int k4 = i % Lq4, rr = i / Lq4, gate = rr & 3, ul = rr >> 2;
    const int row = gate * H + uq_lo + ul;
    const float* src = r < 2 ? p.w_ih + static_cast<size_t>(row) * H + r * Lq + k4 * 4
                             : p.w_hh + static_cast<size_t>(row) * H + (r - 2) * Lq + k4 * 4;
    reinterpret_cast<float4*>(s_wl)[i] = __ldg(reinterpret_cast<const float4*>(src));
  }
  for (int i = tid; i < npq * Hq4; i += kThreads)
    reinterpret_cast<float4*>(s_wp)[i] =
        __ldg(reinterpret_cast<const float4*>(p.w_pred + static_cast<size_t>(pq_lo + i / Hq4) * H + r * Hq) + i % Hq4);
  for (int i = tid; i < njq * Jq4; i += kThreads)
    reinterpret_cast<float4*>(s_wj)[i] =
        __ldg(reinterpret_cast<const float4*>(p.w_out + static_cast<size_t>(jq_lo + i / Jq4) * J + r * Jq) + i % Jq4);
  for (int i = tid; i < nmu * 4; i += kThreads) {
    const int row = (i & 3) * H + uq_lo + mu_lo + (i >> 2);
    s_bl[i] = p.b_ih[row] + p.b_hh[row];
  }
  ctl.init(p);
  // SOS: pending = LSTM(0; 0, 0) = f(bias) for the units this rank finalises; committed state = 0 (hbuf[1] is zeroed)
  for (int i = tid; i < nmu * B; i += kThreads) {
    const int m = i % nmu, b = i / nmu;
    const float* bl = s_bl + m * 4;
    const float c1 = sigmoidf_(bl[0]) * tanhf(bl[2]);
    const float h1 = sigmoidf_(bl[3]) * tanhf(c1);
    s_c[(0 * B + b) * mumax + m] = c1;
    s_c[(1 * B + b) * mumax + m] = 0.f;
    p.hbuf[(static_cast<size_t>(0) * B + b) * H + uq_lo + mu_lo + m] = h1;
  }
  unsigned int bar_target = 0;
  int jbuf = 0, lbuf = 0, pbuf = 0;
  int n_emit, n_active;
  ctl.build_lists(B, &n_emit, &n_active);
  cluster_sync_all();  // every CTA of the cluster is running before the first remote shared-memory store
  grid_sync(p.counter, bar_target);

  bool first = true;
  for (unsigned int it = 0;; ++it) {
    if (!first) {
      // ---- joint at frames t and t + 1 of every active utterance ----------------------------------------------------------------
      if (tid < 2 * kMaxB) s_best[tid] = 0ull;
      __syncthreads();
      for (int s0 = 0; s0 < n_active; s0 += tile_s) {
        const int ns = min(tile_s, n_active - s0), total = ns * Jq4;
        for (int base = 0; base < total; base += kThreads * kJointRound) {
          float4 e0[kJointRound], e1[kJointRound], qq[kJointRound];
#pragma unroll
          for (int u = 0; u < kJointRound; ++u) {
            const int idx = base + u * kThreads + tid;
            if (idx < total) {
              const int bb = ctl.alist[s0 + idx / Jq4], k4 = idx % Jq4, t0 = ctl.t[bb], t1 = min(t0 + 1, ctl.len[bb] - 1);
              e0[u] = __ldg(reinterpret_cast<const float4*>(p.encp + (static_cast<size_t>(bb) * p.T + t0) * J + r * Jq) + k4);
              e1[u] = __ldg(reinterpret_cast<const float4*>(p.encp + (static_cast<size_t>(bb) * p.T + t1) * J + r * Jq) + k4);
              qq[u] = ldcg4(p.predp + static_cast<size_t>(bb) * J + r * Jq + k4 * 4);
            }
          }
#pragma unroll
          for (int u = 0; u < kJointRound; ++u) {
            const int idx = base + u * kThreads + tid;
            if (idx < total) {
              const int i = idx / Jq4, k4 = idx % Jq4;
              float4 z;
              z.x = act_fn(e0[u].x + qq[u].x, p.act), z.y = act_fn(e0[u].y + qq[u].y, p.act);
              z.z = act_fn(e0[u].z + qq[u].z, p.act), z.w = act_fn(e0[u].w + qq[u].w, p.act);
              s_stage[(2 * i) * Jq4 + k4] = z;
              z.x = act_fn(e1[u].x + qq[u].x, p.act), z.y = act_fn(e1[u].y + qq[u].y, p.act);
              z.z = act_fn(e1[u].z + qq[u].z, p.act), z.w = act_fn(e1[u].w + qq[u].w, p.act);
              s_stage[(2 * i + 1) * Jq4 + k4] = z;
            }
          }
        }
        __syncthreads();
        const int nv = 2 * ns, ngroups = (nv + 3) >> 2;
        float* pj = s_pj + jbuf * (kC * 8 * kTileV);
        for (int task = warp; task < ngroups * nchunks; task += kWarps) {
          const int grp = task % ngroups, ch = task / ngroups;
          int zi[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) zi[u] = min(4 * grp + u, nv - 1);
          const float4* wr = reinterpret_cast<const float4*>(s_wj) + ch * 8 * Jq4;
          const float total_k = Jq4 == 40 ? tile_dot_r4<8, -2>(wr, Jq4, njq - ch * 8, s_stage, Jq4, zi, Jq4, lane)
                                          : tile_dot_r4<8, 0>(wr, Jq4, njq - ch * 8, s_stage, Jq4, zi, Jq4, lane);
          const int row = lane >> 2, v = 4 * grp + (lane & 3);  // partial logit of (row, vector) -> the chunk's owner rank
          if (v < nv) st_cluster_f32(pj + (r * 8 + row) * kTileV + v, ch, total_k);
        }
        cluster_sync_all();
        if (r < nchunks && tid < 8 * kTileV) {
          const int row = tid / kTileV, v = tid % kTileV;
          if (v < nv && r * 8 + row < njq) {
            const float* src = pj + row * kTileV + v;
            const float sum = ((src[0] + src[8 * kTileV]) + src[2 * 8 * kTileV]) + src[3 * 8 * kTileV];
            const int out_row = jq_lo + r * 8 + row;
            atomicMax(&s_best[(v & 1) * kMaxB + ctl.alist[s0 + (v >> 1)]], pack_key(sum + __ldg(p.b_out + out_row), out_row));
          }
        }
        jbuf ^= 1;
        __syncthreads();
      }
      if (r < nchunks && tid < 2 * n_active) {
        const int b = ctl.alist[tid >> 1], f = tid & 1;
        atomicMax(&p.slots[((it % 3) * 2 + f) * kMaxB + b], s_best[f * kMaxB + b]);
      }
      grid_sync(p.counter, bar_target);

      // ---- control update (replicated in every CTA) ---------------------------------------------------------------------
      ctl.update(p, it, &n_emit, &n_active);

      // ---- LSTM cell for the utterances that emitted ---------------------------------------------------------------------------
      if (n_emit > 0) {
        for (int s0 = 0; s0 < n_emit; s0 += tile_l) {
          const int ns = min(tile_l, n_emit - s0), total = ns * Lq4;
          for (int base = 0; base < total; base += kThreads * kStageRound) {
            float4 v[kStageRound];
#pragma unroll
            for (int u = 0; u < kStageRound; ++u) {
              const int idx = base + u * kThreads + tid;
              if (idx < total) {
                const int bb = ctl.elist[s0 + idx / Lq4], k4 = idx % Lq4;
                v[u] = r < 2 ? __ldg(reinterpret_cast<const float4*>(p.embed + static_cast<size_t>(ctl.last[bb]) * H + r * Lq) + k4)
                             : ldcg4(p.hbuf + (static_cast<size_t>(ctl.par[bb]) * B + bb) * H + (r - 2) * Lq + k4 * 4);
              }
            }
#pragma unroll
            for (int u = 0; u < kStageRound; ++u) {
              const int idx = base + u * kThreads + tid;
              if (idx < total) s_stage[idx] = v[u];
            }
          }
          __syncthreads();
          const int ngr = (ns + 3) >> 2;
          float* pl = s_pl + lbuf * (kC * mumax * 4 * kTileL);
          for (int task = warp; task < ngr * nuq; task += kWarps) {
            const int grp = task % ngr, ul = task / ngr;
            int zi[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) zi[u] = min(4 * grp + u, ns - 1);
            const float4* wr = reinterpret_cast<const float4*>(s_wl) + static_cast<size_t>(ul) * 4 * Lq4;
            const float total_k = Lq4 == 80 ? tile_dot_r4<4, -3>(wr, Lq4, 4, s_stage, Lq4, zi, Lq4, lane)
                                            : tile_dot_r4<4, 0>(wr, Lq4, 4, s_stage, Lq4, zi, Lq4, lane);
            int owner, m;
            owner_of(ul, nuq, &owner, &m);
            const int gate = (lane >> 2) & 3, sidx = 4 * grp + (lane & 3);
            if (lane < 16 && sidx < ns) st_cluster_f32(pl + ((r * mumax + m) * 4 + gate) * kTileL + sidx, owner, total_k);
          }
          cluster_sync_all();
          if (tid < nmu * kTileL) {
            const int m = tid / kTileL, sidx = tid % kTileL;
            if (sidx < ns) {
              float g4[4];
#pragma unroll
              for (int gate = 0; gate < 4; ++gate) {
                const float* src = pl + (m * 4 + gate) * kTileL + sidx;
                const int st = mumax * 4 * kTileL;
                g4[gate] = (((src[0] + src[st]) + src[2 * st]) + src[3 * st]) + s_bl[m * 4 + gate];
              }
              const int b = ctl.elist[s0 + sidx];
              const int par = ctl.par[b];
              const float c_old = s_c[(par * B + b) * mumax + m];
              const float c_new = sigmoidf_(g4[1]) * c_old + sigmoidf_(g4[0]) * tanhf(g4[2]);
              const float h_new = sigmoidf_(g4[3]) * tanhf(c_new);
              s_c[((par ^ 1) * B + b) * mumax + m] = c_new;
              p.hbuf[(static_cast<size_t>(par ^ 1) * B + b) * H + uq_lo + mu_lo + m] = h_new;
            }
          }
          lbuf ^= 1;
          __syncthreads();
        }
        if (tid < n_emit) ctl.par[ctl.elist[tid]] ^= 1;
        grid_sync(p.counter, bar_target);
      }
      if (n_active == 0) break;
    }
    first = false;

    // ---- joint.pred of the new prediction-network outputs ---------------------------------------------------------------------
    if (n_emit > 0) {
      const int nch4 = (npq + 3) >> 2;
      for (int s0 = 0; s0 < n_emit; s0 += tile_p) {
        const int ns = min(tile_p, n_emit - s0), total = ns * Hq4;
        for (int base = 0; base < total; base += kThreads * kStageRound) {
          float4 v[kStageRound];
#pragma unroll
          for (int u = 0; u < kStageRound; ++u) {
            const int idx = base + u * kThreads + tid;
            if (idx < total) {
              const int bb = ctl.elist[s0 + idx / Hq4];
              v[u] = ldcg4(p.hbuf + (static_cast<size_t>(ctl.par[bb]) * B + bb) * H + r * Hq + (idx % Hq4) * 4);
            }
          }
#pragma unroll
          for (int u = 0; u < kStageRound; ++u) {
            const int idx = base + u * kThreads + tid;
            if (idx < total) s_stage[idx] = v[u];
          }
        }
        __syncthreads();
        const int ngr = (ns + 3) >> 2;
        float* pp = s_pp + pbuf * (kC * mpmax * kTileP);
        for (int task = warp; task < ngr * nch4; task += kWarps) {
          const int grp = task % ngr, ch = task / ngr;
          int zi[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) zi[u] = min(4 * grp + u, ns - 1);
          const float4* wr = reinterpret_cast<const float4*>(s_wp) + ch * 4 * Hq4;
          const float total_k = Hq4 == 40 ? tile_dot_r4<4, -2>(wr, Hq4, npq - ch * 4, s_stage, Hq4, zi, Hq4, lane)
                                          : tile_dot_r4<4, 0>(wr, Hq4, npq - ch * 4, s_stage, Hq4, zi, Hq4, lane);
          const int row = ch * 4 + ((lane >> 2) & 3), sidx = 4 * grp + (lane & 3);
          if (lane < 16 && row < npq && sidx < ns) {
            int owner, m;
            owner_of(row, npq, &owner, &m);
            st_cluster_f32(pp + (r * mpmax + m) * kTileP + sidx, owner, total_k);
          }
        }
        cluster_sync_all();
        if (tid < nmp * kTileP) {
          const int m = tid / kTileP, sidx = tid % kTileP;
          if (sidx < ns) {
            const float* src = pp + m * kTileP + sidx;
            const int st = mpmax * kTileP, row = pq_lo + mp_lo + m;
            p.predp[static_cast<size_t>(ctl.elist[s0 + sidx]) * J + row] =
                (((src[0] + src[st]) + src[2 * st]) + src[3 * st]) + __ldg(p.b_pred + row);
          }
        }
        pbuf ^= 1;
        __syncthreads();
      }
      grid_sync(p.counter, bar_target);
    }
    if (n_active == 0) break;
  }

  ctl.write_results(p, s_c, mumax, uq_lo + mu_lo, nmu);
  cluster_sync_all();  // no CTA of the cluster exits while a sibling could still address its shared memory
}

struct RnntScratch {
  size_t sync_off, sync_bytes, hbuf_off, hbuf_bytes, predp_off;
  RnntEncScratch enc;
};
RnntScratch rnnt_scratch_layout(int E, int H, int J, int B, int T) {
  RnntScratch s;
  const int Bc = B < kMaxB ? B : kMaxB;
  size_t off = 0;
  s.sync_off = off;
  s.sync_bytes = align256(512 + sizeof(unsigned long long) * 3 * 2 * kMaxB);  // barrier counter | slots from byte 512 on
  off += s.sync_bytes;
  s.hbuf_off = off;
  s.hbuf_bytes = align256(sizeof(float) * 2 * Bc * H);
  off += s.hbuf_bytes;
  s.predp_off = off;
  off += align256(sizeof(float) * Bc * J);
  s.enc = rnnt_enc_scratch(off, E, J, B, T);
  return s;
}

// dynamic shared memory without the staging buffer
size_t rnnt_smem_fixed_bytes(int H, int J, int V1, int G, int B, int* umax, int* pmax, int* jmax) {
  *umax = (H + G - 1) / G;
  *pmax = (J + G - 1) / G;
  *jmax = (V1 + G - 1) / G;
  return sizeof(float) * (static_cast<size_t>(*umax) * 4 * 2 * H + static_cast<size_t>(*pmax) * H + static_cast<size_t>(*jmax) * J +
                          static_cast<size_t>(*umax) * 4 + (static_cast<size_t>(2) * B * *umax + 3) / 4 * 4);
}

// cluster variant: dynamic shared memory without the staging buffer (rows per CLUSTER in umax / pmax / jmax)
size_t rnnt_c4_fixed_bytes(int H, int J, int V1, int NQ, int B, int* umax, int* pmax, int* jmax) {
  *umax = (H + NQ - 1) / NQ;
  *pmax = (J + NQ - 1) / NQ;
  *jmax = (V1 + NQ - 1) / NQ;
  const size_t mumax = (*umax + kC - 1) / kC, mpmax = (*pmax + kC - 1) / kC;
  return sizeof(float) * (static_cast<size_t>(*umax) * 4 * (H / 2) + static_cast<size_t>(*pmax) * (H / 4) +
                          static_cast<size_t>(*jmax) * (J / 4) + mumax * 4 + (static_cast<size_t>(2) * B * mumax + 3) / 4 * 4 +
                          static_cast<size_t>(2) * kC * 8 * kTileV + static_cast<size_t>(2) * kC * mumax * 4 * kTileL +
                          (static_cast<size_t>(2) * kC * mpmax * kTileP + 3) / 4 * 4);
}

// Launch configuration of rnnt_greedy_c4_kernel: clusters of kC CTAs and, for the launch itself (not the occupancy
// query), the cooperative attribute.
cudaLaunchConfig_t c4_launch_config(int grid, size_t smem, cudaStream_t st, bool cooperative, cudaLaunchAttribute (&attr)[2]) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kC;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeCooperative;
  attr[1].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = cooperative ? 2 : 1;
  return cfg;
}

// Plans the cluster variant: number of co-resident clusters, shared-memory split.  Returns false when it is not asked for
// or the device / the sizes rule it out (the row-partitioned kernel is used then).
bool g_c4_unusable = false;  // set when a cooperative cluster launch was refused once (the other kernel serves from then on)

bool rnnt_c4_plan(int H, int J, int V1, int Bmax, int max_smem, RnntParams* p, int* grid, size_t* smem) {
  // The default.  Measured (32 / 64 / 128 utterances x 500 frames): 11.3 / 17.2 / 29.5 ms against 12.1 / 19.1 / 32.8 ms for the
  // row-partitioned kernel.  Nsight Compute cannot replay a cooperative cluster launch (it aborts the process with
  // LaunchFailed), so the row-partitioned kernel is selected FOR PROFILING: when ncu has injected itself into the process
  // (it exports NV_COMPUTE_PROFILER_PERFWORKS_DIR to its target, profiles/r5f_ncu_env_probe.log) or with CFB_RNNT_CLUSTER=0.
  const char* env = getenv("CFB_RNNT_CLUSTER");
  const bool profiler_attached = getenv("NV_COMPUTE_PROFILER_PERFWORKS_DIR") != nullptr;
  const bool want = env != nullptr ? atoi(env) != 0 : !profiler_attached;
  if (!want || g_c4_unusable || (H % 16) || (J % 16)) return false;
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, rnnt_greedy_c4_kernel) != cudaSuccess) return false;
  const size_t budget = static_cast<size_t>(max_smem) - fa.sharedSizeBytes;
  if (cudaFuncSetAttribute(rnnt_greedy_c4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(budget)) != cudaSuccess)
    return false;
  cudaLaunchAttribute attr[2];
  const cudaLaunchConfig_t cfg = c4_launch_config(kC * 64, budget, 0, false, attr);
  int nq = 0;
  if (cudaOccupancyMaxActiveClusters(&nq, rnnt_greedy_c4_kernel, &cfg) != cudaSuccess || nq < 8) {
    cudaGetLastError();
    return false;
  }
  const size_t fixed = rnnt_c4_fixed_bytes(H, J, V1, nq, Bmax, &p->umax, &p->pmax, &p->jmax);
  if ((p->jmax + 7) / 8 > kC) return false;  // more 8-row output chunks per cluster than ranks to finalise them
  const size_t need = sizeof(float) * static_cast<size_t>(4) * (H / 2 > 2 * (J / 4) ? H / 2 : 2 * (J / 4));
  if (budget < fixed + need) return false;
  size_t useful = static_cast<size_t>(kTileV) * (J / 4);
  if (static_cast<size_t>(kTileL) * (H / 2) > useful) useful = static_cast<size_t>(kTileL) * (H / 2);
  if (static_cast<size_t>(kTileP) * (H / 4) > useful) useful = static_cast<size_t>(kTileP) * (H / 4);
  useful *= sizeof(float);
  const size_t stage = (budget - fixed < useful ? budget - fixed : useful) / 16 * 16;
  p->stage_floats = static_cast<int>(stage / sizeof(float));
  *grid = nq * kC;
  *smem = fixed + stage;
  return true;
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

}  // namespace

bool rnnt_weights_valid(const cfb_rnnt_weights& w, int x_dtype) {
  const int E = w.enc_hidden, H = w.pred_hidden, J = w.joint_hidden;
  return E >= 8 && E % 8 == 0 && H >= 4 && H % 4 == 0 && J >= 4 && J % 4 == 0 && w.num_classes_with_blank >= 2 &&
         w.activation >= 0 && w.activation <= 2 && (x_dtype == CFB_F32 || x_dtype == CFB_BF16) && w.embed && w.w_ih && w.w_hh &&
         w.b_ih && w.b_hh && w.w_pred && w.b_pred && w.w_enc && w.b_enc && w.w_out && w.b_out;
}

int rnnt_device_query(int* sms, int* max_smem) {
  int dev = 0, coop = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return CFB_ERR_CUDA;
  cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
  return !coop || *sms < 1 ? CFB_ERR_UNSUPPORTED : CFB_OK;
}

// On the tensor cores with split operands: A' = [hi | hi | lo] (fp32 input) or [x | x] (bf16), W' = [hi | lo | hi].
int rnnt_joint_enc(const cfb_rnnt_weights& w, const void* encoded, int x_dtype, int B, int T, uint8_t* ws, const RnntEncScratch& s,
                   cudaStream_t st) {
  const int E = w.enc_hidden, J = w.joint_hidden;
  const bool xf32 = x_dtype == CFB_F32;
  const long long M = static_cast<long long>(B) * T;
  bf16* a_split = reinterpret_cast<bf16*>(ws + s.a_off);
  bf16* w_split = reinterpret_cast<bf16*>(ws + s.w_off);
  const long long n = M * E;
  const int blocks = static_cast<int>((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16);
  split_bf16_kernel<<<blocks, 256, 0, st>>>(encoded, a_split, M, E, xf32 ? 0 : 2);
  split_bf16_kernel<<<(J * E + 255) / 256, 256, 0, st>>>(w.w_enc, w_split, J, E, 1);
  GemmDesc g;
  g.A = a_split;
  g.lda = xf32 ? 3 * E : 2 * E;
  g.W = w_split;
  g.ldw = 3 * E;
  g.M = static_cast<int>(M);
  g.N = J;
  g.K = xf32 ? 3 * E : 2 * E;
  g.epi = EPI_LINEAR;
  g.out_bf16 = false;
  g.ep.bias = w.b_enc;
  g.ep.out = reinterpret_cast<float*>(ws + s.encp_off);
  g.ep.ldo = J;
  std::string err;
  return launch_gemm_tc(g, st, &err) != 0 ? CFB_ERR_CUDA : CFB_OK;
}

}  // namespace cfb

using namespace cfb;

extern "C" {

size_t cfb_rnnt_greedy_scratch_bytes(int enc_hidden, int pred_hidden, int joint_hidden, int B, int T) {
  if (enc_hidden < 1 || pred_hidden < 1 || joint_hidden < 1 || B < 1 || T < 1) return 0;
  return rnnt_scratch_layout(enc_hidden, pred_hidden, joint_hidden, B, T).enc.end;
}

int cfb_op_rnnt_greedy(const cfb_rnnt_weights* w, const void* encoded, int x_dtype, const int32_t* encoded_len, int B, int T,
                       int max_symbols, int max_tokens, int32_t* tokens, int32_t* timesteps, int32_t* n_tokens, float* scores,
                       float* h_out, float* c_out, int32_t* flags, void* scratch, size_t scratch_bytes, cfb_stream stream) {
  if (!w || !encoded || !encoded_len || !tokens || !timesteps || !n_tokens || !scores || !h_out || !c_out || !flags || !scratch)
    return CFB_ERR_INVALID_ARG;
  if (B < 1 || T < 1 || max_tokens < 1 || !rnnt_weights_valid(*w, x_dtype)) return CFB_ERR_INVALID_ARG;
  const int E = w->enc_hidden, H = w->pred_hidden, J = w->joint_hidden, V1 = w->num_classes_with_blank;
  const RnntScratch lay = rnnt_scratch_layout(E, H, J, B, T);
  if (scratch_bytes < lay.enc.end || (reinterpret_cast<uintptr_t>(scratch) & 255)) return CFB_ERR_WORKSPACE;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>(scratch);

  int sms = 0, max_smem = 0;
  if (int rc = rnnt_device_query(&sms, &max_smem)) return rc;
  RnntParams p = {};
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, rnnt_greedy_kernel) != cudaSuccess) return CFB_ERR_CUDA;
  // shared memory: my weight rows + cell states + as much activation staging as is useful and fits
  const int Bmax = B < kMaxB ? B : kMaxB;
  int grid = sms;
  size_t smem = 0;
  bool clustered = false;
  auto plan = [&]() -> int {
    clustered = rnnt_c4_plan(H, J, V1, Bmax, max_smem, &p, &grid, &smem);
    if (clustered) return CFB_OK;
    grid = sms;
    const size_t fixed = rnnt_smem_fixed_bytes(H, J, V1, sms, Bmax, &p.umax, &p.pmax, &p.jmax);
    const size_t room = static_cast<size_t>(max_smem) > fixed + fa.sharedSizeBytes ? max_smem - fixed - fa.sharedSizeBytes : 0;
    const size_t useful = sizeof(float) * static_cast<size_t>(Bmax < kMaxTile ? (Bmax + 3) / 4 * 4 : kMaxTile) * (2 * H > J ? 2 * H : J);
    const size_t need = sizeof(float) * static_cast<size_t>(4) * (2 * H > J ? 2 * H : J);  // one group of 4 utterances
    if (room < need) return CFB_ERR_UNSUPPORTED;  // weights do not fit on chip
    const size_t stage = (room < useful ? room : useful) / 16 * 16;
    p.stage_floats = static_cast<int>(stage / sizeof(float));
    smem = fixed + stage;
    if (cudaFuncSetAttribute(rnnt_greedy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess)
      return CFB_ERR_CUDA;
    return CFB_OK;
  };
  if (int rc = plan()) return rc;
  if (int rc = rnnt_joint_enc(*w, encoded, x_dtype, B, T, ws, lay.enc, st)) return rc;

  const float* encp = reinterpret_cast<const float*>(ws + lay.enc.encp_off);
  for (int b0 = 0; b0 < B; b0 += kMaxB) {
    const int Bc = B - b0 < kMaxB ? B - b0 : kMaxB;
    if (cudaMemsetAsync(ws + lay.sync_off, 0, lay.sync_bytes + lay.hbuf_bytes, st) != cudaSuccess) return CFB_ERR_CUDA;
    p.E = E, p.H = H, p.J = J, p.V1 = V1, p.act = w->activation, p.B = Bc, p.T = T;
    p.max_symbols = max_symbols, p.max_tokens = max_tokens;
    p.embed = w->embed, p.w_ih = w->w_ih, p.w_hh = w->w_hh, p.b_ih = w->b_ih, p.b_hh = w->b_hh;
    p.w_pred = w->w_pred, p.b_pred = w->b_pred, p.w_out = w->w_out, p.b_out = w->b_out;
    p.encp = encp + static_cast<size_t>(b0) * T * J;
    p.lens = encoded_len + b0;
    p.counter = reinterpret_cast<unsigned int*>(ws + lay.sync_off);
    p.slots = reinterpret_cast<unsigned long long*>(ws + lay.sync_off + 512);
    p.hbuf = reinterpret_cast<float*>(ws + lay.hbuf_off);
    p.predp = reinterpret_cast<float*>(ws + lay.predp_off);
    p.tokens = tokens + static_cast<size_t>(b0) * max_tokens;
    p.timesteps = timesteps + static_cast<size_t>(b0) * max_tokens;
    p.n_tokens = n_tokens + b0;
    p.scores = scores + b0;
    p.h_out = h_out + static_cast<size_t>(b0) * H;
    p.c_out = c_out + static_cast<size_t>(b0) * H;
    p.flags = flags;
    if (clustered) {
      cudaLaunchAttribute attr[2];
      const cudaLaunchConfig_t cfg = c4_launch_config(grid, smem, st, true, attr);
      if (cudaLaunchKernelEx(&cfg, rnnt_greedy_c4_kernel, p) != cudaSuccess) {
        cudaGetLastError();      // refused (e.g. the clusters are not co-resident right now): nothing was enqueued
        g_c4_unusable = true;
        if (int rc = plan()) return rc;
      }
    }
    if (!clustered) {
      void* args[] = {&p};
      if (cudaLaunchCooperativeKernel(reinterpret_cast<void*>(rnnt_greedy_kernel), dim3(grid), dim3(kThreads), args, smem, st) !=
          cudaSuccess)
        return CFB_ERR_CUDA;
    }
  }
  return cudaGetLastError() == cudaSuccess ? CFB_OK : CFB_ERR_CUDA;
}

}  // extern "C"
