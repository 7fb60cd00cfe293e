// Transducer beam search on the encoder output (decoding.strategy = beam, search_type = default): the prediction network
// and joint of rnnt_greedy.cu and the hypothesis bookkeeping of BeamRNNTInfer.default_beam_search / greedy_search
// (parts/submodules/rnnt_beam_decoding.py; restated in oracle/rnnt_beam_oracle.py) as ONE persistent cooperative kernel.
//
// The reference decodes one utterance at a time on the host and synchronises once per hypothesis expansion.  Here
//   * joint.enc is applied to every frame up front by the split-operand tcgen05 GEMM (as in the greedy decode),
//   * one CTA per SM keeps ITS rows of the LSTM, joint.pred and output-layer weights in shared memory in fp32,
//   * utterances advance in lock-step iterations; in each one every active utterance expands exactly one hypothesis, the
//     maximum of its `hyps` list, so the reference's order of operations is kept.  An iteration has four phases, each
//     ended by a grid barrier:
//       A  LSTM cell of the popped prefix-tree nodes whose prediction-network output is not computed yet (my hidden units),
//       B  joint.pred of those nodes (my rows),
//       C  the joint at (frame, node) of every active utterance (my output rows) -> logits in global memory,
//       D  control, on the CTA that owns the utterance (CTA b owns utterance b of the launch): fp32 log-softmax over the
//          V + 1 classes, top-beam_k non-blank candidates (first index on ties, like torch.topk on distinct values),
//          fp64 score updates, the break test, the frame advance, the next pick and, at the end, the n-best sort.
//     A and B are skipped in an iteration where no popped node needs them: a node's prediction-network output is computed
//     once (the reference's cache keyed by the label sequence) and kept in a state slot for every later expansion.
//   * Each utterance owns a prefix-tree node arena (token, parent, frame, depth, state slot) and state slots (h, c, g) in
//     global scratch; its `hyps` / `kept` lists (fp64 score, node) live in the owner CTA's shared memory, in the
//     reference's list order (the max pick and the stable sort depend on it).
//   * Capacities (nodes, state slots, expansions per frame, list entries, output length) are parameters.  An utterance
//     that would exceed one sets flag bit 0 and stops cleanly; the caller decodes again with larger capacities.
#include <float.h>
#include <stdlib.h>

#include "../../include/cfb.h"
#include "common.cuh"
#include "rnnt_common.cuh"

namespace cfb {
namespace {

constexpr int kThreads = 512;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxB = 128;        // utterances per launch (one owner CTA each)
constexpr int kMaxBeamK = 64;     // non-blank candidates per expansion
constexpr int kGreedyMaxSymbols = 5;  // greedy_search's symbols per frame (beam_size == 1)
constexpr int kWork = 8;          // ints per utterance in the work record
constexpr int kMaxHyps = 4 * kThreads;  // list entries (the list shift moves up to 4 entries per thread)
// flags: bit 0 = some capacity was exceeded; the other bits say which one
constexpr int kFlagExpansions = 2, kFlagHyps = 4, kFlagNodes = 8, kFlagStates = 16, kFlagLen = 32;

// work record of utterance b, written by its owner in phase D, read by every CTA after the barrier
enum { W_ACTIVE = 0, W_NEED = 1, W_SLOT = 2, W_PSLOT = 3, W_TOKEN = 4, W_FRAME = 5 };

struct BeamParams {
  int E, H, J, V1, act, B, T, beam, beam_k, score_norm, greedy;
  float temperature;
  int max_nodes, max_states, max_expansions, max_hyps, max_len;
  const float *embed, *w_ih, *w_hh, *b_ih, *b_hh, *w_pred, *b_pred, *w_out, *b_out;
  const float* encp;         // (B*T, J) = joint.enc(encoded)
  const int32_t* lens;
  unsigned int* counter;     // grid barrier
  int* work;                 // [kMaxB][kWork]
  float* logits;             // [B][V1]
  int4* nodes;               // [B][max_nodes] (token, parent, frame, state slot)
  int* depth;                // [B][max_nodes]
  float* states;             // [B][max_states][2H + J]  (h, c, g)
  // outputs (rows of this launch)
  int32_t *n_hyps, *lengths, *tokens, *timesteps, *stats, *flags;
  double* scores;
  float *h_out, *c_out;
  int umax, pmax, jmax, stage_floats;
};

__device__ __forceinline__ float warp_dot(const float* __restrict__ w, const float* __restrict__ z, int K4, int lane) {
  const float4* w4 = reinterpret_cast<const float4*>(w);
  const float4* z4 = reinterpret_cast<const float4*>(z);
  float acc = 0.f;
  for (int k4 = lane; k4 < K4; k4 += 32) acc = dot4(w4[k4], z4[k4], acc);
  return warp_sum(acc);
}

// block-wide reductions (every thread gets the result); fixed order, so results do not depend on timing
__device__ float block_max_f(float v, float* s_red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = s_red[0];
  for (int i = 1; i < kWarps; ++i) r = fmaxf(r, s_red[i]);
  return r;
}
__device__ float block_sum_f(float v, float* s_red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = s_red[0];
  for (int i = 1; i < kWarps; ++i) r += s_red[i];
  return r;
}
__device__ unsigned long long block_max_u64(unsigned long long v, unsigned long long* s_red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
    v = w > v ? w : v;
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  unsigned long long r = s_red[0];
  for (int i = 1; i < kWarps; ++i) r = s_red[i] > r ? s_red[i] : r;
  return r;
}
// first maximal element of a list of doubles: (score, index) with the larger score, the smaller index on equal scores
__device__ int block_argmax_first(const double* s, int n, double* s_redd, int* s_redi) {
  double best = -DBL_MAX;
  int bi = 0x7fffffff;
  for (int i = threadIdx.x; i < n; i += kThreads)
    if (s[i] > best) best = s[i], bi = i;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) best = ob, bi = oi;
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_redd[threadIdx.x >> 5] = best, s_redi[threadIdx.x >> 5] = bi;
  __syncthreads();
  best = s_redd[0], bi = s_redi[0];
  for (int i = 1; i < kWarps; ++i)
    if (s_redd[i] > best || (s_redd[i] == best && s_redi[i] < bi)) best = s_redd[i], bi = s_redi[i];
  return bi;
}

__global__ void __launch_bounds__(kThreads, 1) rnnt_beam_kernel(const BeamParams p) {
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = gridDim.x, cta = blockIdx.x;
  const int H = p.H, J = p.J, V1 = p.V1, B = p.B, K2 = 2 * p.H, SW = 2 * p.H + p.J;
  const int blank = V1 - 1;

  int u_lo, u_hi, p_lo, p_hi, j_lo, j_hi;
  row_range(H, cta, G, &u_lo, &u_hi);
  row_range(J, cta, G, &p_lo, &p_hi);
  row_range(V1, cta, G, &j_lo, &j_hi);
  const int nu = u_hi - u_lo, np = p_hi - p_lo, nj = j_hi - j_lo;

  // ---- shared memory: weights of my rows, the staging buffer, the owned utterance's hypothesis lists ---------------------
  float* s_wl = smem;                                          // [umax][4][2H]
  float* s_wp = s_wl + static_cast<size_t>(p.umax) * 4 * K2;   // [pmax][H]
  float* s_wj = s_wp + static_cast<size_t>(p.pmax) * H;        // [jmax][J]
  float* s_bl = s_wj + static_cast<size_t>(p.jmax) * J;        // [umax][4]
  float* s_stage = s_bl + ((p.umax * 4 + 3) / 4) * 4;          // [stage_floats]
  double* s_hs = reinterpret_cast<double*>(s_stage + ((p.stage_floats + 1) / 2) * 2);  // hyps scores [max_hyps]
  double* s_ks = s_hs + p.max_hyps;                             // kept scores
  int* s_hn = reinterpret_cast<int*>(s_ks + p.max_hyps);        // hyps nodes
  int* s_kn = s_hn + p.max_hyps;                                // kept nodes
  __shared__ int s_wk[kMaxB][kWork];
  __shared__ int s_alist[kMaxB], s_nlist[kMaxB];
  __shared__ int s_na, s_nn;
  __shared__ float s_redf[kWarps];
  __shared__ unsigned long long s_redu[kWarps];
  __shared__ double s_redd[kWarps];
  __shared__ int s_redi[kWarps];
  __shared__ float s_cv[kMaxBeamK];
  __shared__ int s_ck[kMaxBeamK];
  // control of the owned utterance (thread 0 writes, the block reads after a barrier)
  __shared__ int c_t, c_len, c_sym, c_nh, c_nk, c_nodes, c_states, c_pops, c_cur, c_done, c_pops_total, c_pops_max, c_why;
  __shared__ double c_score;

  load_row_weights(p, u_lo, nu, p_lo, np, j_lo, nj, s_wl, s_bl, s_wp, s_wj);

  const int b_own = cta < B ? cta : -1;
  int4* nodes = b_own >= 0 ? p.nodes + static_cast<size_t>(b_own) * p.max_nodes : nullptr;
  int* depth = b_own >= 0 ? p.depth + static_cast<size_t>(b_own) * p.max_nodes : nullptr;
  float* states = b_own >= 0 ? p.states + static_cast<size_t>(b_own) * p.max_states * SW : nullptr;

  // Writes the n-best list of the owned utterance (kept, sorted by sort_nbest), its statistics, and ends it.
  auto finish = [&](bool overflow) {
    __syncthreads();
    const int n = overflow ? 0 : c_nk, b = b_own;
    // sort_nbest: stable descending sort by score / len(y) (score_norm) or score; ranks instead of a sequential sort
    for (int i = tid; i < n; i += kThreads) {
      const int nd = s_kn[i];
      const double si = s_ks[i];
      const double ki = p.score_norm ? si / static_cast<double>(depth[nd] + 1) : si;
      int rank = 0;
      for (int j = 0; j < n; ++j) {
        const double kj = p.score_norm ? s_ks[j] / static_cast<double>(depth[s_kn[j]] + 1) : s_ks[j];
        rank += (kj > ki) || (kj == ki && j < i);
      }
      const size_t row = static_cast<size_t>(b) * p.max_expansions + rank;
      const int skip = p.greedy ? 1 : 0;  // greedy_search's y has no leading blank, its timestep no -1
      const int len = depth[nd] + 1 - skip;
      p.scores[row] = si;
      p.lengths[row] = len;
      if (len > p.max_len) {
        atomicOr(p.flags, 1 | kFlagLen);
      } else {
        int cur = nd;
        for (int pos = len - 1; pos >= 0; --pos) {
          const int4 e = nodes[cur];
          p.tokens[row * p.max_len + pos] = e.x;
          p.timesteps[row * p.max_len + pos] = e.z;
          cur = e.y;
        }
      }
    }
    // final state of each hypothesis: the state its last label is predicted from (zeros for the initial hypothesis)
    for (int i = tid; i < n * H; i += kThreads) {
      const int r = i / H, u = i % H, nd = s_kn[r];
      const double si = s_ks[r];
      const double ki = p.score_norm ? si / static_cast<double>(depth[nd] + 1) : si;
      int rank = 0;
      for (int j = 0; j < n; ++j) {
        const double kj = p.score_norm ? s_ks[j] / static_cast<double>(depth[s_kn[j]] + 1) : s_ks[j];
        rank += (kj > ki) || (kj == ki && j < r);
      }
      const int par = nodes[nd].y;
      const int ps = par >= 0 ? nodes[par].w : -1;
      const size_t row = static_cast<size_t>(b) * p.max_expansions + rank;
      p.h_out[row * H + u] = ps >= 0 ? __ldcg(states + static_cast<size_t>(ps) * SW + u) : 0.f;
      p.c_out[row * H + u] = ps >= 0 ? __ldcg(states + static_cast<size_t>(ps) * SW + H + u) : 0.f;
    }
    if (tid == 0) {
      if (overflow) atomicOr(p.flags, 1 | c_why);
      p.n_hyps[b] = n;
      p.stats[b * 4 + 0] = c_pops_total;
      p.stats[b * 4 + 1] = c_nodes;
      p.stats[b * 4 + 2] = c_states;
      p.stats[b * 4 + 3] = c_pops_max;
      c_done = 1;
      p.work[b * kWork + W_ACTIVE] = 0;
    }
    __syncthreads();
  };

  // Pops the first maximal hypothesis of `hyps` and publishes the work record for it (thread 0 decides, then barrier).
  auto pop_best = [&]() {
    __syncthreads();
    const int i = (p.greedy || c_nh == 0) ? -1 : block_argmax_first(s_hs, c_nh, s_redd, s_redi);
    double sc = 0.0;
    int nd = 0;
    if (i >= 0) sc = s_hs[i], nd = s_hn[i];
    __syncthreads();
    if (i >= 0) {  // hyps.remove(best): shift the tail left by one (read all, barrier, write all)
      double vs[4];
      int vn[4];
      int cnt = 0;
      for (int j = i + 1 + tid; j < c_nh && cnt < 4; j += kThreads, ++cnt) vs[cnt] = s_hs[j], vn[cnt] = s_hn[j];
      __syncthreads();
      cnt = 0;
      for (int j = i + 1 + tid; j < c_nh && cnt < 4; j += kThreads, ++cnt) s_hs[j - 1] = vs[cnt], s_hn[j - 1] = vn[cnt];
    }
    __syncthreads();
    if (tid == 0) {
      bool overflow = false;
      if (i >= 0) {
        --c_nh;
        c_cur = nd;
        c_score = sc;
      }
      nd = c_cur;
      if (++c_pops > p.max_expansions) overflow = true, c_why |= kFlagExpansions;
      c_pops_total += 1;
      c_pops_max = max(c_pops_max, c_pops);
      int4 e = nodes[nd];
      int need = 0;
      if (!overflow && e.w < 0) {  // prediction-network output not computed for this label sequence yet: take a slot
        if (c_states >= p.max_states) {
          overflow = true;
          c_why |= kFlagStates;
        } else {
          e.w = c_states++;
          nodes[nd] = e;
          need = 1;
        }
      }
      int* w = p.work + b_own * kWork;
      if (overflow) {
        c_done = 2;
      } else {
        w[W_NEED] = need;
        w[W_SLOT] = e.w;
        w[W_PSLOT] = e.y >= 0 ? nodes[e.y].w : -1;
        w[W_TOKEN] = e.x;
        w[W_FRAME] = c_t;
        w[W_ACTIVE] = 1;
      }
    }
    __syncthreads();
    if (c_done == 2) finish(true);
  };

  if (b_own >= 0) {
    if (tid == 0) {
      c_len = min(max(p.lens[b_own], 0), p.T);
      c_t = 0, c_sym = 0, c_nh = 0, c_nk = 0, c_pops = 0, c_pops_total = 0, c_pops_max = 0, c_done = 0, c_why = 0;
      c_score = 0.0;
      nodes[0] = make_int4(blank, -1, -1, -1);  // the initial hypothesis: y = [blank], timestep = [-1]
      depth[0] = 0;
      c_nodes = 1, c_states = 0, c_cur = 0;
      if (c_len == 0) {  // nothing to decode: the initial hypothesis is the result
        s_ks[0] = 0.0, s_kn[0] = 0, c_nk = 1;
      }
    }
    __syncthreads();
    if (c_len == 0) {
      if (p.greedy) {  // greedy_search returns its empty hypothesis
        if (tid == 0) {
          p.n_hyps[b_own] = 1;
          p.scores[static_cast<size_t>(b_own) * p.max_expansions] = 0.0;
          p.lengths[static_cast<size_t>(b_own) * p.max_expansions] = 0;
          for (int i = 0; i < 4; ++i) p.stats[b_own * 4 + i] = 0;
          p.work[b_own * kWork + W_ACTIVE] = 0;
          c_done = 1;
        }
        __syncthreads();
      } else {
        finish(false);
      }
    } else {
      pop_best();  // the initial hypothesis (hyps is empty: the pick keeps c_cur = 0)
    }
  }
  unsigned int bar_target = 0;
  grid_sync(p.counter, bar_target);

  for (;;) {
    // ---- the work records of this iteration (identical in every CTA) --------------------------------------------------
    for (int i = tid; i < B * kWork; i += kThreads) s_wk[i / kWork][i % kWork] = __ldcg(p.work + i);
    __syncthreads();
    if (tid == 0) {
      int na = 0, nn = 0;
      for (int b = 0; b < B; ++b)
        if (s_wk[b][W_ACTIVE]) {
          s_alist[na++] = b;
          if (s_wk[b][W_NEED]) s_nlist[nn++] = b;
        }
      s_na = na, s_nn = nn;
    }
    __syncthreads();
    const int n_active = s_na, n_need = s_nn;
    if (n_active == 0) break;

    if (n_need > 0) {
      // ---- A: LSTM cell of the new nodes, my hidden units ----------------------------------------------------------------
      const int tile = min(kMaxB, p.stage_floats / K2);
      for (int s0 = 0; nu > 0 && s0 < n_need; s0 += tile) {
        const int ns = min(tile, n_need - s0);
        for (int i = tid; i < ns * (K2 / 4); i += kThreads) {  // stage [embed(token) | h of the parent's state]
          const int b = s_nlist[s0 + i / (K2 / 4)], k4 = i % (K2 / 4), ps = s_wk[b][W_PSLOT];
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (k4 < H / 4) {
            if (s_wk[b][W_TOKEN] != blank) v = __ldg(reinterpret_cast<const float4*>(p.embed + static_cast<size_t>(s_wk[b][W_TOKEN]) * H) + k4);
          } else if (ps >= 0) {
            v = ldcg4(p.states + (static_cast<size_t>(b) * p.max_states + ps) * SW + (k4 - H / 4) * 4);
          }
          reinterpret_cast<float4*>(s_stage)[i] = v;
        }
        __syncthreads();
        for (int task = warp; task < nu * ns; task += kWarps) {
          const int ul = task / ns, u = task % ns, b = s_nlist[s0 + u];
          const float* z = s_stage + static_cast<size_t>(u) * K2;
          float g4[4];
#pragma unroll
          for (int gate = 0; gate < 4; ++gate)
            g4[gate] = warp_dot(s_wl + (static_cast<size_t>(ul) * 4 + gate) * K2, z, K2 / 4, lane) + s_bl[ul * 4 + gate];
          if (lane == 0) {
            const int ps = s_wk[b][W_PSLOT];
            const float c_old = ps >= 0 ? __ldcg(p.states + (static_cast<size_t>(b) * p.max_states + ps) * SW + H + u_lo + ul) : 0.f;
            const float c_new = sigmoidf_(g4[1]) * c_old + sigmoidf_(g4[0]) * tanhf(g4[2]);
            const float h_new = sigmoidf_(g4[3]) * tanhf(c_new);
            float* st = p.states + (static_cast<size_t>(b) * p.max_states + s_wk[b][W_SLOT]) * SW;
            st[u_lo + ul] = h_new;
            st[H + u_lo + ul] = c_new;
          }
        }
        __syncthreads();
      }
      grid_sync(p.counter, bar_target);
      // ---- B: joint.pred of the new nodes, my rows ----------------------------------------------------------------------
      const int tile_p = min(kMaxB, p.stage_floats / H);
      for (int s0 = 0; np > 0 && s0 < n_need; s0 += tile_p) {
        const int ns = min(tile_p, n_need - s0);
        for (int i = tid; i < ns * (H / 4); i += kThreads) {
          const int b = s_nlist[s0 + i / (H / 4)];
          reinterpret_cast<float4*>(s_stage)[i] =
              ldcg4(p.states + (static_cast<size_t>(b) * p.max_states + s_wk[b][W_SLOT]) * SW + (i % (H / 4)) * 4);
        }
        __syncthreads();
        for (int task = warp; task < np * ns; task += kWarps) {
          const int r = task / ns, u = task % ns, b = s_nlist[s0 + u];
          const float acc = warp_dot(s_wp + static_cast<size_t>(r) * H, s_stage + static_cast<size_t>(u) * H, H / 4, lane);
          if (lane == 0)
            p.states[(static_cast<size_t>(b) * p.max_states + s_wk[b][W_SLOT]) * SW + K2 + p_lo + r] = acc + __ldg(p.b_pred + p_lo + r);
        }
        __syncthreads();
      }
      grid_sync(p.counter, bar_target);
    }

    // ---- C: joint logits of my output rows for every active utterance at (frame, popped node) -----------------------------
    const int tile_j = min(kMaxB, p.stage_floats / J);
    for (int s0 = 0; nj > 0 && s0 < n_active; s0 += tile_j) {
      const int ns = min(tile_j, n_active - s0);
      for (int i = tid; i < ns * (J / 4); i += kThreads) {
        const int b = s_alist[s0 + i / (J / 4)], k4 = i % (J / 4);
        const float4 e = __ldg(reinterpret_cast<const float4*>(p.encp + (static_cast<size_t>(b) * p.T + s_wk[b][W_FRAME]) * J) + k4);
        const float4 q = ldcg4(p.states + (static_cast<size_t>(b) * p.max_states + s_wk[b][W_SLOT]) * SW + K2 + k4 * 4);
        float4 z;
        z.x = act_fn(e.x + q.x, p.act), z.y = act_fn(e.y + q.y, p.act), z.z = act_fn(e.z + q.z, p.act), z.w = act_fn(e.w + q.w, p.act);
        reinterpret_cast<float4*>(s_stage)[i] = z;
      }
      __syncthreads();
      for (int task = warp; task < nj * ns; task += kWarps) {
        const int r = task / ns, u = task % ns, b = s_alist[s0 + u];
        const float acc = warp_dot(s_wj + static_cast<size_t>(r) * J, s_stage + static_cast<size_t>(u) * J, J / 4, lane);
        if (lane == 0) p.logits[static_cast<size_t>(b) * V1 + j_lo + r] = acc + __ldg(p.b_out + j_lo + r);
      }
      __syncthreads();
    }
    grid_sync(p.counter, bar_target);

    // ---- D: control of the owned utterance ------------------------------------------------------------------------------
    if (b_own >= 0 && s_wk[b_own][W_ACTIVE]) {
      float* lp = s_stage;  // log-probabilities of the V + 1 classes
      float m = -FLT_MAX;
      for (int i = tid; i < V1; i += kThreads) {
        const float v = __ldcg(p.logits + static_cast<size_t>(b_own) * V1 + i) / p.temperature;
        lp[i] = v;
        m = fmaxf(m, v);
      }
      m = block_max_f(m, s_redf);
      float s = 0.f;
      for (int i = tid; i < V1; i += kThreads) s += expf(lp[i] - m);
      const float logs = logf(block_sum_f(s, s_redf));
      for (int i = tid; i < V1; i += kThreads) lp[i] = (lp[i] - m) - logs;
      __syncthreads();
      // candidates: greedy -> the arg-max over all V + 1 classes; beam -> the top beam_k non-blank classes, best first
      const int nc = p.greedy ? 1 : p.beam_k, lim = p.greedy ? V1 : V1 - 1;
      unsigned long long prev = ~0ull;
      for (int r = 0; r < nc; ++r) {
        unsigned long long key = 0ull;
        for (int i = tid; i < lim; i += kThreads) {
          const unsigned long long k = pack_key(lp[i], i);
          if (k < prev && k > key) key = k;
        }
        key = block_max_u64(key, s_redu);
        prev = key;
        if (tid == 0) unpack_key(key, &s_cv[r], &s_ck[r]);
      }
      __syncthreads();
      if (p.greedy) {
        if (tid == 0) {
          const int k = s_ck[0];
          bool end = false, overflow = false;
          if (k == blank) {
            c_sym = 0;
            end = ++c_t >= c_len;
          } else {
            if (c_nodes >= p.max_nodes) {
              overflow = true;
              c_why |= kFlagNodes;
            } else {
              c_score += static_cast<double>(s_cv[0]);
              const int nd = c_nodes++;
              nodes[nd] = make_int4(k, c_cur, c_t, -1);
              depth[nd] = depth[c_cur] + 1;
              c_cur = nd;
              if (++c_sym >= kGreedyMaxSymbols) {
                c_sym = 0;
                end = ++c_t >= c_len;
              }
            }
          }
          if (!overflow && (k == blank || c_sym == 0)) c_pops = 0;  // a new frame
          if (end) s_ks[0] = c_score, s_kn[0] = c_cur, c_nk = 1;
          c_done = overflow ? 2 : (end ? 3 : 0);
        }
        __syncthreads();
        if (c_done == 2) finish(true);
        else if (c_done == 3) finish(false);
        else pop_best();
      } else {
        if (tid == 0) {  // the beam_k + 1 extensions of the popped hypothesis, in the reference's order
          const bool nodes_full = c_nodes + p.beam_k > p.max_nodes;
          const bool lists_full = c_nh + p.beam_k > p.max_hyps || c_nk + 1 > p.max_hyps;
          c_why |= (nodes_full ? kFlagNodes : 0) | (lists_full ? kFlagHyps : 0);
          const bool overflow = nodes_full || lists_full;
          if (!overflow) {
            for (int r = 0; r < p.beam_k; ++r) {
              const int nd = c_nodes++;
              nodes[nd] = make_int4(s_ck[r], c_cur, c_t, -1);
              depth[nd] = depth[c_cur] + 1;
              s_hs[c_nh] = c_score + static_cast<double>(s_cv[r]);
              s_hn[c_nh++] = nd;
            }
            s_ks[c_nk] = c_score + static_cast<double>(lp[blank]);
            s_kn[c_nk++] = c_cur;
          }
          c_done = overflow ? 2 : 0;
        }
        __syncthreads();
        if (c_done == 2) {
          finish(true);
        } else {
          // break test: the kept hypotheses above the best of hyps, stably sorted ascending, if there are >= beam of them
          double hm = -DBL_MAX;
          for (int i = tid; i < c_nh; i += kThreads) hm = fmax(hm, s_hs[i]);
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) hm = fmax(hm, __shfl_xor_sync(0xffffffffu, hm, o));
          __syncthreads();
          if (lane == 0) s_redd[warp] = hm;
          __syncthreads();
          hm = s_redd[0];
          for (int i = 1; i < kWarps; ++i) hm = fmax(hm, s_redd[i]);
          if (tid == 0) {  // kept holds at most one entry per expansion of this frame: counted sequentially
            int cnt = 0;
            for (int i = 0; i < c_nk; ++i) cnt += s_ks[i] > hm;
            s_redi[0] = cnt;
          }
          __syncthreads();
          const int cnt = s_redi[0];
          if (cnt >= p.beam) {
            // kept = most; hyps = kept for the next frame: ranks of a stable ascending sort, written straight into hyps
            for (int i = tid; i < c_nk; i += kThreads) {
              const double si = s_ks[i];
              if (!(si > hm)) continue;
              int rank = 0;
              for (int j = 0; j < c_nk; ++j) {
                const double sj = s_ks[j];
                rank += sj > hm && (sj < si || (sj == si && j < i));
              }
              s_hs[rank] = si;
              s_hn[rank] = s_kn[i];
            }
            __syncthreads();
            if (tid == 0) {
              c_t += 1;
              c_pops = 0;
              c_nh = cnt;
            }
            __syncthreads();
            if (c_t >= c_len) {  // the last frame: the n-best list is `most`
              for (int i = tid; i < cnt; i += kThreads) s_ks[i] = s_hs[i], s_kn[i] = s_hn[i];
              __syncthreads();
              if (tid == 0) c_nk = cnt;
              finish(false);
            } else {
              if (tid == 0) c_nk = 0;
              pop_best();
            }
          } else {
            pop_best();
          }
        }
      }
    }
    grid_sync(p.counter, bar_target);
  }
}

struct BeamScratch {
  size_t sync_off, sync_bytes, work_off, logits_off, nodes_off, depth_off, states_off;
  RnntEncScratch enc;
};
BeamScratch beam_scratch_layout(int E, int H, int J, int V1, int B, int T, const cfb_rnnt_beam_caps& c) {
  BeamScratch s;
  const size_t Bc = B < kMaxB ? B : kMaxB;
  size_t off = 0;
  s.sync_off = off;
  s.sync_bytes = 512;
  off += s.sync_bytes;
  s.work_off = off;
  off += align256(sizeof(int) * kMaxB * kWork);
  s.logits_off = off;
  off += align256(sizeof(float) * Bc * V1);
  s.nodes_off = off;
  off += align256(sizeof(int4) * Bc * c.max_nodes);
  s.depth_off = off;
  off += align256(sizeof(int) * Bc * c.max_nodes);
  s.states_off = off;
  off += align256(sizeof(float) * Bc * c.max_states * (2 * static_cast<size_t>(H) + J));
  s.enc = rnnt_enc_scratch(off, E, J, B, T);
  return s;
}

bool caps_valid(const cfb_rnnt_beam_caps* c) {
  return c && c->max_expansions >= 1 && c->max_nodes >= 1 && c->max_states >= 1 && c->max_hyps >= 1 && c->max_len >= 1;
}

}  // namespace
}  // namespace cfb

using namespace cfb;

extern "C" {

size_t cfb_rnnt_beam_scratch_bytes(int enc_hidden, int pred_hidden, int joint_hidden, int num_classes_with_blank, int B, int T,
                                   const cfb_rnnt_beam_caps* caps) {
  if (enc_hidden < 1 || pred_hidden < 1 || joint_hidden < 1 || num_classes_with_blank < 2 || B < 1 || T < 1 || !caps_valid(caps))
    return 0;
  return beam_scratch_layout(enc_hidden, pred_hidden, joint_hidden, num_classes_with_blank, B, T, *caps).enc.end;
}

int cfb_op_rnnt_beam(const cfb_rnnt_weights* w, const void* encoded, int x_dtype, const int32_t* encoded_len, int B, int T,
                     int beam_size, int score_norm, float temperature, const cfb_rnnt_beam_caps* caps, int32_t* n_hyps,
                     int32_t* lengths, int32_t* tokens, int32_t* timesteps, double* scores, float* h_out, float* c_out,
                     int32_t* stats, int32_t* flags, void* scratch, size_t scratch_bytes, cfb_stream stream) {
  if (!w || !encoded || !encoded_len || !n_hyps || !lengths || !tokens || !timesteps || !scores || !h_out || !c_out || !stats ||
      !flags || !scratch || !caps_valid(caps))
    return CFB_ERR_INVALID_ARG;
  if (B < 1 || T < 1 || beam_size < 1 || !(temperature > 0.f) || !rnnt_weights_valid(*w, x_dtype)) return CFB_ERR_INVALID_ARG;
  const int E = w->enc_hidden, H = w->pred_hidden, J = w->joint_hidden, V1 = w->num_classes_with_blank;
  const int V = V1 - 1;
  const int beam = beam_size < V1 ? beam_size : V1, beam_k = beam < V ? beam : V;  // default_beam_search's widths
  if (beam_k > kMaxBeamK || caps->max_hyps > kMaxHyps) return CFB_ERR_UNSUPPORTED;
  const BeamScratch lay = beam_scratch_layout(E, H, J, V1, B, T, *caps);
  if (scratch_bytes < lay.enc.end || (reinterpret_cast<uintptr_t>(scratch) & 255)) return CFB_ERR_WORKSPACE;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>(scratch);

  int sms = 0, max_smem = 0;
  if (int rc = rnnt_device_query(&sms, &max_smem)) return rc;
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, rnnt_beam_kernel) != cudaSuccess) return CFB_ERR_CUDA;
  // shared memory: my weight rows + the owned utterance's two hypothesis lists + as much staging as is useful and fits
  BeamParams p = {};
  const int G = sms;
  p.umax = (H + G - 1) / G, p.pmax = (J + G - 1) / G, p.jmax = (V1 + G - 1) / G;
  const size_t fixed = sizeof(float) * (static_cast<size_t>(p.umax) * 4 * 2 * H + static_cast<size_t>(p.pmax) * H +
                                        static_cast<size_t>(p.jmax) * J + (p.umax * 4 + 3) / 4 * 4) +
                       static_cast<size_t>(caps->max_hyps) * 2 * (sizeof(double) + sizeof(int)) + 16;
  const size_t room = static_cast<size_t>(max_smem) > fixed + fa.sharedSizeBytes ? max_smem - fixed - fa.sharedSizeBytes : 0;
  const int Bl = B < kMaxB ? (B < G ? B : G) : (kMaxB < G ? kMaxB : G);  // utterances per launch (one owner CTA each)
  const size_t widest = static_cast<size_t>(2 * H > J ? 2 * H : J);
  const size_t need = sizeof(float) * (widest > static_cast<size_t>(V1) ? widest : static_cast<size_t>(V1));
  const size_t useful = sizeof(float) * widest * (Bl < 16 ? Bl : 16);
  if (room < need) return CFB_ERR_UNSUPPORTED;  // weights (or the lists) do not fit on chip
  size_t stage = room < (useful > need ? useful : need) ? room : (useful > need ? useful : need);
  stage = stage / 16 * 16;
  p.stage_floats = static_cast<int>(stage / sizeof(float));
  const size_t smem = fixed + stage;
  if (cudaFuncSetAttribute(rnnt_beam_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess)
    return CFB_ERR_CUDA;

  if (int rc = rnnt_joint_enc(*w, encoded, x_dtype, B, T, ws, lay.enc, st)) return rc;

  const float* encp = reinterpret_cast<const float*>(ws + lay.enc.encp_off);
  const int X = caps->max_expansions;
  for (int b0 = 0; b0 < B; b0 += Bl) {
    const int Bc = B - b0 < Bl ? B - b0 : Bl;
    if (cudaMemsetAsync(ws + lay.sync_off, 0, lay.sync_bytes, st) != cudaSuccess) return CFB_ERR_CUDA;
    p.E = E, p.H = H, p.J = J, p.V1 = V1, p.act = w->activation, p.B = Bc, p.T = T;
    p.beam = beam, p.beam_k = beam_k, p.score_norm = score_norm != 0, p.greedy = beam_size == 1, p.temperature = temperature;
    p.max_nodes = caps->max_nodes, p.max_states = caps->max_states, p.max_expansions = X, p.max_hyps = caps->max_hyps;
    p.max_len = caps->max_len;
    p.embed = w->embed, p.w_ih = w->w_ih, p.w_hh = w->w_hh, p.b_ih = w->b_ih, p.b_hh = w->b_hh;
    p.w_pred = w->w_pred, p.b_pred = w->b_pred, p.w_out = w->w_out, p.b_out = w->b_out;
    p.encp = encp + static_cast<size_t>(b0) * T * J;
    p.lens = encoded_len + b0;
    p.counter = reinterpret_cast<unsigned int*>(ws + lay.sync_off);
    p.work = reinterpret_cast<int*>(ws + lay.work_off);
    p.logits = reinterpret_cast<float*>(ws + lay.logits_off);
    p.nodes = reinterpret_cast<int4*>(ws + lay.nodes_off);
    p.depth = reinterpret_cast<int*>(ws + lay.depth_off);
    p.states = reinterpret_cast<float*>(ws + lay.states_off);
    p.n_hyps = n_hyps + b0;
    p.lengths = lengths + static_cast<size_t>(b0) * X;
    p.tokens = tokens + static_cast<size_t>(b0) * X * caps->max_len;
    p.timesteps = timesteps + static_cast<size_t>(b0) * X * caps->max_len;
    p.scores = scores + static_cast<size_t>(b0) * X;
    p.h_out = h_out + static_cast<size_t>(b0) * X * H;
    p.c_out = c_out + static_cast<size_t>(b0) * X * H;
    p.stats = stats + static_cast<size_t>(b0) * 4;
    p.flags = flags;
    void* args[] = {&p};
    if (cudaLaunchCooperativeKernel(reinterpret_cast<void*>(rnnt_beam_kernel), dim3(G), dim3(kThreads), args, smem, st) != cudaSuccess)
      return CFB_ERR_CUDA;
  }
  return cudaGetLastError() == cudaSuccess ? CFB_OK : CFB_ERR_CUDA;
}

}  // extern "C"
