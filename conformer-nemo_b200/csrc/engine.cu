// Host side of the cfb library: handle, weight ingestion + packing, workspace planning, the forward schedule and the
// C ABI of include/cfb.h.  The forward pass is enqueue-only: no allocation, no synchronisation, one stream.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include <cuda_fp16.h>
#include <nvtx3/nvToolsExt.h>  // header-only NVTX v3: ranges are no-ops unless a profiler injected itself

#include <algorithm>

#include "../../include/cfb.h"
#include "common.cuh"

using namespace cfb;

namespace {

struct HostTensor {
  std::vector<float> data;
  std::vector<int64_t> shape;
  int64_t numel() const {
    int64_t n = 1;
    for (auto s : shape) n *= s;
    return n;
  }
};

// device arena entry: offset in bytes
struct Slot {
  size_t off = 0;
};

struct LayerW {
  // LayerNorm affine (fp32): ff1, att, conv, ff2, out
  Slot ln_g[5], ln_b[5];
  Slot ff_w1[2], ff_b1[2], ff_w2[2], ff_b2[2];
  Slot w_qkv, b_qkv, b_qv, w_out, b_out;
  Slot w_pw1, b_pw1, dw_taps, dw_bias, dw_taps32, w_pw2, b_pw2;
};

std::string g_create_error;

}  // namespace

struct cfb_handle {
  cfb_config cfg;
  int device = 0;
  bool validate = false;  // CFB_PREC_FP32_VALIDATE
  // derived
  int d = 0, C = 0, F0 = 0, F1 = 0, F2 = 0, Fh = 0, dff = 0, H = 0, dk = 0, dkp = 64, Dp = 0, L = 0, ksize = 0;
  int d_out = 0;
  bool has_out_proj = false;
  std::map<std::string, HostTensor> staged;
  bool finalized = false;
  // device arena
  uint8_t* arena = nullptr;
  size_t arena_bytes = 0;
  Slot sub_w1, sub_b1, sub_w1g, sub_w2, sub_b2, sub_w3, sub_b3, w_pos, div_term, w_oproj, b_oproj;
  std::vector<LayerW> layers;
  int sms = 0;  // streaming multiprocessors of the device
  int launches = 0;
  // a batch may run as up to kMaxGroups parts (run_parts): part 0 on the caller's stream, part g on group_stream[g]
  static constexpr int kMaxGroups = 4;
  cudaStream_t group_stream[kMaxGroups] = {};
  cudaEvent_t ev_fork = nullptr, group_join[kMaxGroups] = {};
  mutable std::string err;
  // optional per-launch event timing
  bool profiling = false;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  struct Rec {
    const char* label;
    size_t e0, e1;
  };
  std::vector<Rec> recs;

  size_t esz() const { return validate ? 4 : 2; }  // bytes per activation / matrix element
  template <typename T>
  T* at(const Slot& s) const {
    return reinterpret_cast<T*>(arena + s.off);
  }
};

namespace {

int fail(const cfb_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  return code;
}

size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

int conv_out(int n) { return (n - 1) / 2 + 1; }  // k=3, s=2, p=1 (n >= 1)

// a named region of the workspace
struct Region {
  size_t off = 0, bytes = 0;
};

struct Plan {
  int B, T, T1, T2, Th, N, P;  // P = 2*T2-1
  Region y1, y2, x, a, hbuf, qkv, ctx, g, c, pe, pos, a0, raw, cols;
  Region tables;  // packed batches only: the PackedTables arrays
  size_t total;
};

// Layout of a packed batch, computed from host-side lengths with the integer arithmetic packed_plan_kernel uses.
struct PackedShape {
  int n_rows = 0;   // token rows over all slots
  int n_tiles = 0;  // attention query tiles
  int t2_max = 0;   // dense output extent T' of the padded batch
  int first = 0, step = 1, count = 0;  // the group of utterances first, first + step, ... (count of them) this layout holds
};
PackedShape packed_shape(const int64_t* lengths_host, int B, int T, int first = 0, int step = 1) {
  PackedShape ps;
  ps.t2_max = conv_out(conv_out(T));
  ps.first = first;
  ps.step = step;
  for (int b = first; b < B; b += step) {
    ++ps.count;
    long long len = lengths_host ? lengths_host[b] : T;
    len = len < 0 ? 0 : (len > T ? T : len);
    const int t1 = static_cast<int>((len + 1) >> 1);
    const int t2 = (t1 + 1) >> 1;
    const int rows = packed_slot_rows(t2);
    ps.n_rows += rows;
    ps.n_tiles += (rows + 127) / 128;
  }
  return ps;
}

// Workspace layout of the dense (B, T) batch, or with pk of the packed group pk: one virtual sequence of 4 * pk->n_rows
// input frames (common.cuh, PackedTables) whose positional table covers pk->t2_max frames.
Plan make_plan(const cfb_handle* h, int B, int T, const PackedShape* pk = nullptr) {
  Plan p{};
  if (pk) {
    B = 1;
    T = 4 * pk->n_rows;
  }
  p.B = B;
  p.T = T;
  p.T1 = conv_out(T);
  p.T2 = conv_out(p.T1);
  p.Th = (p.T1 + 1) / 2;
  p.N = B * p.T2;
  p.P = 2 * (pk ? pk->t2_max : p.T2) - 1;
  const size_t e = h->esz();
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const Region r{off, bytes};
    off = align_up(off + bytes);
    return r;
  };
  const size_t N = static_cast<size_t>(p.N);
  p.y1 = take(static_cast<size_t>(B) * 4 * p.Th * h->Fh * h->C * e);
  p.y2 = take(N * h->F2 * h->C * e);
  p.x = take(N * h->d * 4);
  p.a = take(N * h->d * e);
  p.hbuf = take(N * h->dff * e);
  p.qkv = take(N * 4 * h->Dp * e);
  p.ctx = take(N * h->Dp * e);
  p.g = take(N * h->d * e);
  p.c = take(N * h->d * e);
  p.pe = take(static_cast<size_t>(p.P) * h->d * e);
  p.pos = take(static_cast<size_t>(p.P) * h->L * h->Dp * e);
  if (!h->validate) {
    p.a0 = take(static_cast<size_t>(B) * 4 * p.Th * h->Fh * kConv0Cols * 2);  // first conv's GEMM operand
  } else {
    size_t raw = N * h->dff;
    raw = std::max(raw, N * 3 * h->Dp);
    raw = std::max(raw, static_cast<size_t>(p.P) * h->L * h->Dp);
    raw = std::max(raw, N * h->F2 * h->C);
    raw = std::max(raw, N * 2 * h->d);
    raw = std::max(raw, N * static_cast<size_t>(std::max(h->d_out, h->d)));
    p.raw = take(raw * 4);
    p.cols = take(N * h->F2 * 9 * h->C * 4);
  }
  if (pk)
    p.tables = take((static_cast<size_t>(2) * pk->count + 2 * N + N / kPackAlign + 8) * 4 + static_cast<size_t>(pk->n_tiles) * 16 + 64);
  p.total = off;
  return p;
}

PackedTables carve_tables(uint8_t* base, int B, int n_rows) {
  PackedTables t;
  int32_t* q = reinterpret_cast<int32_t*>(base);
  t.seq_row0 = q, q += B;
  t.seq_rows = q, q += B;
  t.row_t = q, q += n_rows;
  t.row_out = q, q += n_rows;
  t.blk_seq = q, q += n_rows / kPackAlign;
  t.tiles = reinterpret_cast<int4*>((reinterpret_cast<uintptr_t>(q) + 15) & ~uintptr_t(15));
  return t;
}

// cfb_forward runs a bf16 batch of B >= 8 as two half-batches on two streams (micro-batching)
int dense_parts(const cfb_handle* h, int B) { return (!h->validate && B >= 8) ? 2 : 1; }
// utterances [first, first + count) of part i when a dense batch of B runs as n contiguous parts
struct Range {
  int first, count;
};
Range dense_part(int B, int n, int i) {
  const int per = (B + n - 1) / n;
  return {i * per, std::min(per, B - i * per)};
}

// A batch split into n parts lays the parts' plans end to end in the workspace.  The workspace a call needs is the
// largest such sum over the splits n = 1 .. max_parts it may take; plan(n, i) is the plan of part i of n.
template <typename PartPlan>
size_t workspace_need(int max_parts, PartPlan plan) {
  size_t need = 0;
  for (int n = 1; n <= max_parts; ++n) {
    size_t sum = 0;
    for (int i = 0; i < n; ++i) sum += plan(n, i).total;
    need = std::max(need, sum);
  }
  return need;
}
size_t dense_workspace(const cfb_handle* h, int B, int T) {
  return workspace_need(dense_parts(h, B), [&](int n, int i) { return make_plan(h, dense_part(B, n, i).count, T); });
}
// any group count up to min(B, kMaxGroups): CFB_PACKED_GROUPS can force each of them
size_t packed_workspace(const cfb_handle* h, const int64_t* lengths_host, int B, int T) {
  return workspace_need(std::min(B, cfb_handle::kMaxGroups), [&](int n, int i) {
    const PackedShape ps = packed_shape(lengths_host, B, T, i, n);
    return make_plan(h, B, T, &ps);
  });
}

const HostTensor* find(const cfb_handle* h, const std::string& key) {
  auto it = h->staged.find(key);
  return it == h->staged.end() ? nullptr : &it->second;
}

bool shape_is(const HostTensor* t, std::initializer_list<int64_t> want) {
  if (!t || t->shape.size() != want.size()) return false;
  size_t i = 0;
  for (auto w : want)
    if (t->shape[i++] != w) return false;
  return true;
}

// arena builder: host-side image + slots
struct ArenaBuilder {
  std::vector<uint8_t> img;
  Slot put_f32(const std::vector<float>& v) {
    Slot s;
    s.off = align_up(img.size());
    img.resize(s.off + v.size() * 4);
    memcpy(img.data() + s.off, v.data(), v.size() * 4);
    return s;
  }
  Slot put_mat(const std::vector<float>& v, bool as_f32) {
    if (as_f32) return put_f32(v);
    Slot s;
    s.off = align_up(img.size());
    img.resize(s.off + v.size() * 2);
    bf16* dst = reinterpret_cast<bf16*>(img.data() + s.off);
    for (size_t i = 0; i < v.size(); ++i) dst[i] = __float2bfloat16_rn(v[i]);
    return s;
  }
};

}  // namespace

// =====================================================================================================================
extern "C" {

const char* cfb_last_error(const cfb_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int cfb_create(const cfb_config* cfg, int device, cfb_handle** out) {
  if (!cfg || !out) {
    g_create_error = "cfb_create: null argument";
    return CFB_ERR_INVALID_ARG;
  }
  *out = nullptr;
  auto bad = [&](int code, const std::string& m) {
    g_create_error = "cfb_create: " + m;
    return code;
  };
  if (cfg->feat_in < 1 || cfg->n_layers < 1 || cfg->d_model < 16 || cfg->n_heads < 1 || cfg->ff_expansion_factor < 1)
    return bad(CFB_ERR_INVALID_ARG, "feat_in, n_layers, d_model, n_heads and ff_expansion_factor must be positive");
  if (cfg->feat_in > kMaxFeatIn)
    return bad(CFB_ERR_UNSUPPORTED, "feat_in > " + std::to_string(kMaxFeatIn) +
                                        " is not supported (the first conv stages (feat_in + 2) x 34 fp32 features of a block in 48 KB of shared memory)");
  if (cfg->d_model % cfg->n_heads) return bad(CFB_ERR_INVALID_ARG, "d_model must be divisible by n_heads");
  if (cfg->subsampling_factor != 4)
    return bad(CFB_ERR_UNSUPPORTED, "only subsampling_factor=4 (two strided convolutions) is supported");
  if (cfg->d_model % 16) return bad(CFB_ERR_UNSUPPORTED, "d_model must be a multiple of 16");
  if (cfg->d_model > 1024) return bad(CFB_ERR_UNSUPPORTED, "d_model > 1024 is not supported");
  if (cfg->d_model / cfg->n_heads > 128) return bad(CFB_ERR_UNSUPPORTED, "head dimension > 128 is not supported");
  if ((cfg->d_model / cfg->n_heads) % 2) return bad(CFB_ERR_UNSUPPORTED, "head dimension must be even");
  if (cfg->conv_kernel_size < 1 || cfg->conv_kernel_size > 31 || cfg->conv_kernel_size % 2 == 0)
    return bad(CFB_ERR_UNSUPPORTED, "conv_kernel_size must be odd and <= 31");
  const int C = cfg->subsampling_conv_channels == -1 ? cfg->d_model : cfg->subsampling_conv_channels;
  if (C < 8 || C % 8) return bad(CFB_ERR_UNSUPPORTED, "subsampling_conv_channels must be a multiple of 8");
  if (cfg->precision != CFB_PREC_BF16 && cfg->precision != CFB_PREC_FP32_VALIDATE)
    return bad(CFB_ERR_INVALID_ARG, "unknown precision");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev)
    return bad(CFB_ERR_CUDA, "no such CUDA device (this library has no CPU fallback)");
  cudaDeviceProp prop{};
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10) return bad(CFB_ERR_UNSUPPORTED, "the kernels are built for sm_100a (Blackwell B200) only");

  cfb_handle* h = new cfb_handle();
  h->cfg = *cfg;
  h->device = device;
  h->sms = prop.multiProcessorCount;
  h->validate = cfg->precision == CFB_PREC_FP32_VALIDATE;
  h->d = cfg->d_model;
  h->C = C;
  h->F0 = cfg->feat_in;
  h->F1 = conv_out(h->F0);
  h->F2 = conv_out(h->F1);
  h->Fh = (h->F1 + 1) / 2;
  h->dff = cfg->d_model * cfg->ff_expansion_factor;
  h->H = cfg->n_heads;
  h->dk = h->d / h->H;
  h->dkp = h->dk <= 64 ? 64 : 128;  // every head padded to the width of its attention kernel (attention_tc.cu / _tc128.cu)
  h->Dp = h->H * h->dkp;
  h->L = cfg->n_layers;
  h->ksize = cfg->conv_kernel_size;
  h->has_out_proj = cfg->feat_out > 0 && cfg->feat_out != cfg->d_model;
  h->d_out = h->has_out_proj ? cfg->feat_out : h->d;
  if (h->dff % 8 || h->d_out % 8) {
    delete h;
    return bad(CFB_ERR_UNSUPPORTED, "d_ff and feat_out must be multiples of 8");
  }
  cudaSetDevice(device);
  bool ok = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) == cudaSuccess;
  for (int g = 1; ok && g < cfb_handle::kMaxGroups; ++g)
    ok = cudaStreamCreateWithFlags(&h->group_stream[g], cudaStreamNonBlocking) == cudaSuccess &&
         cudaEventCreateWithFlags(&h->group_join[g], cudaEventDisableTiming) == cudaSuccess;
  if (!ok) {
    cfb_destroy(h);
    return bad(CFB_ERR_CUDA, "could not create the group streams / events");
  }
  *out = h;
  return CFB_OK;
}

void cfb_destroy(cfb_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->arena) cudaFree(h->arena);
  for (int g = 1; g < cfb_handle::kMaxGroups; ++g) {
    if (h->group_stream[g]) cudaStreamDestroy(h->group_stream[g]);
    if (h->group_join[g]) cudaEventDestroy(h->group_join[g]);
  }
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  for (auto& e : h->ev_pool) cudaEventDestroy(e);
  delete h;
}

int cfb_set_weight(cfb_handle* h, const char* ref_key, const void* ptr, int dtype, const int64_t* shape, int ndim) {
  if (!h) return CFB_ERR_INVALID_ARG;
  if (!ref_key || !ptr || ndim < 0 || ndim > 8 || (ndim > 0 && !shape))
    return fail(h, CFB_ERR_INVALID_ARG, "cfb_set_weight: null argument");
  const std::string key(ref_key);
  const std::string tail = "num_batches_tracked";
  if (key.size() >= tail.size() && key.compare(key.size() - tail.size(), tail.size(), tail) == 0) return CFB_OK;
  HostTensor t;
  int64_t n = 1;
  for (int i = 0; i < ndim; ++i) {
    if (shape[i] < 0) return fail(h, CFB_ERR_INVALID_ARG, "cfb_set_weight: negative dimension for " + key);
    t.shape.push_back(shape[i]);
    n *= shape[i];
  }
  t.data.resize(static_cast<size_t>(n));
  cudaSetDevice(h->device);
  cudaError_t e = cudaSuccess;
  if (dtype == CFB_F32) {
    e = cudaMemcpy(t.data.data(), ptr, static_cast<size_t>(n) * 4, cudaMemcpyDefault);
  } else if (dtype == CFB_BF16 || dtype == CFB_F16) {
    std::vector<uint16_t> tmp(static_cast<size_t>(n));
    e = cudaMemcpy(tmp.data(), ptr, static_cast<size_t>(n) * 2, cudaMemcpyDefault);
    if (e == cudaSuccess) {
      for (int64_t i = 0; i < n; ++i) {
        if (dtype == CFB_BF16) {
          uint32_t u = static_cast<uint32_t>(tmp[i]) << 16;
          memcpy(&t.data[i], &u, 4);
        } else {
          __half hv;
          memcpy(&hv, &tmp[i], 2);
          t.data[i] = __half2float(hv);
        }
      }
    }
  } else {
    return fail(h, CFB_ERR_INVALID_ARG, "cfb_set_weight: dtype must be f32, bf16 or f16 for " + key);
  }
  if (e != cudaSuccess) return fail(h, CFB_ERR_CUDA, std::string("cfb_set_weight: copy failed: ") + cudaGetErrorString(e));
  h->staged[key] = std::move(t);
  h->finalized = false;
  return CFB_OK;
}

int cfb_finalize_weights(cfb_handle* h) {
  if (!h) return CFB_ERR_INVALID_ARG;
  const int d = h->d, C = h->C, F2 = h->F2, dff = h->dff, H = h->H, dk = h->dk, dkp = h->dkp, Dp = h->Dp, L = h->L;
  const int ks = h->ksize;
  const bool f32 = h->validate;
  std::string missing;
  auto need = [&](const std::string& key, std::initializer_list<int64_t> shape) -> const HostTensor* {
    const HostTensor* t = find(h, key);
    if (!t) {
      if (missing.empty()) missing = "missing weight: " + key;
      return nullptr;
    }
    if (!shape_is(t, shape)) {
      if (missing.empty()) {
        missing = "bad shape for " + key + ": got (";
        for (auto s : t->shape) missing += std::to_string(s) + ",";
        missing += ") expected (";
        for (auto s : shape) missing += std::to_string(s) + ",";
        missing += ")";
      }
      return nullptr;
    }
    return t;
  };

  ArenaBuilder ab;
  // ---- subsampling (subsampling.py:99-116,160)
  const HostTensor* c0w = need("pre_encode.conv.0.weight", {C, 1, 3, 3});
  const HostTensor* c0b = need("pre_encode.conv.0.bias", {C});
  const HostTensor* c2w = need("pre_encode.conv.2.weight", {C, C, 3, 3});
  const HostTensor* c2b = need("pre_encode.conv.2.bias", {C});
  const HostTensor* ow = need("pre_encode.out.weight", {d, static_cast<int64_t>(C) * F2});
  const HostTensor* ob = need("pre_encode.out.bias", {d});
  if (!missing.empty()) return fail(h, CFB_ERR_MISSING_WEIGHT, "cfb_finalize_weights: " + missing);
  h->sub_w1 = ab.put_f32(c0w->data);
  h->sub_b1 = ab.put_f32(c0b->data);
  {
    // (C x 24) bf16 weight of the GEMM form of the first conv: [w (9) | w (9) | bias_hi | bias_lo | 0 x 4]
    std::vector<float> w(static_cast<size_t>(C) * kConv0Cols, 0.f);
    for (int n = 0; n < C; ++n) {
      for (int q = 0; q < 9; ++q) w[static_cast<size_t>(n) * kConv0Cols + q] = w[static_cast<size_t>(n) * kConv0Cols + 9 + q] = c0w->data[n * 9 + q];
      const float bh = __bfloat162float(__float2bfloat16_rn(c0b->data[n]));
      w[static_cast<size_t>(n) * kConv0Cols + 18] = bh;
      w[static_cast<size_t>(n) * kConv0Cols + 19] = c0b->data[n] - bh;
    }
    h->sub_w1g = ab.put_mat(w, false);
  }
  {
    std::vector<float> w(static_cast<size_t>(C) * 9 * C);
    for (int n = 0; n < C; ++n)
      for (int c = 0; c < C; ++c)
        for (int t = 0; t < 9; ++t)
          w[(static_cast<size_t>(n) * 9 + t) * C + c] = c2w->data[(static_cast<size_t>(n) * C + c) * 9 + t];
    h->sub_w2 = ab.put_mat(w, f32);
    h->sub_b2 = ab.put_f32(c2b->data);
  }
  {
    // fold x * sqrt(d_model) (multi_head_attention.py:305-306) and permute K from (c, f) to (f, c)
    const float xs = h->cfg.xscaling ? sqrtf(static_cast<float>(d)) : 1.f;
    std::vector<float> w(static_cast<size_t>(d) * F2 * C), b(d);
    for (int n = 0; n < d; ++n) {
      for (int c = 0; c < C; ++c)
        for (int f = 0; f < F2; ++f)
          w[(static_cast<size_t>(n) * F2 + f) * C + c] = ow->data[static_cast<size_t>(n) * C * F2 + c * F2 + f] * xs;
      b[n] = ob->data[n] * xs;
    }
    h->sub_w3 = ab.put_mat(w, f32);
    h->sub_b3 = ab.put_f32(b);
  }
  // ---- sinusoid frequencies (multi_head_attention.py:238-241)
  {
    std::vector<float> div(d / 2);
    const HostTensor* dt = find(h, "pos_enc.div_term");
    if (dt && dt->numel() == d / 2) {
      div = dt->data;
    } else {
      const float cst = static_cast<float>(-(log(10000.0) / d));
      for (int m = 0; m < d / 2; ++m) div[m] = expf(static_cast<float>(2 * m) * cst);
    }
    h->div_term = ab.put_f32(div);
  }
  // ---- layers
  h->layers.assign(L, LayerW());
  std::vector<float> wpos(static_cast<size_t>(L) * Dp * d, 0.f);
  static const char* ln_names[5] = {"norm_feed_forward1", "norm_self_att", "norm_conv", "norm_feed_forward2", "norm_out"};
  for (int l = 0; l < L && missing.empty(); ++l) {
    const std::string p = "layers." + std::to_string(l) + ".";
    LayerW& lw = h->layers[l];
    for (int i = 0; i < 5; ++i) {
      const HostTensor* g = need(p + ln_names[i] + ".weight", {d});
      const HostTensor* b = need(p + ln_names[i] + ".bias", {d});
      if (!g || !b) break;
      lw.ln_g[i] = ab.put_f32(g->data);
      lw.ln_b[i] = ab.put_f32(b->data);
    }
    for (int f = 0; f < 2 && missing.empty(); ++f) {
      const std::string q = p + (f == 0 ? "feed_forward1." : "feed_forward2.");
      const HostTensor* w1 = need(q + "linear1.weight", {dff, d});
      const HostTensor* b1 = need(q + "linear1.bias", {dff});
      const HostTensor* w2 = need(q + "linear2.weight", {d, dff});
      const HostTensor* b2 = need(q + "linear2.bias", {d});
      if (!w1 || !b1 || !w2 || !b2) break;
      lw.ff_w1[f] = ab.put_mat(w1->data, f32);
      lw.ff_b1[f] = ab.put_f32(b1->data);
      lw.ff_w2[f] = ab.put_mat(w2->data, f32);
      lw.ff_b2[f] = ab.put_f32(b2->data);
    }
    if (!missing.empty()) break;
    const std::string a = p + "self_attn.";
    const HostTensor* wq = need(a + "linear_q.weight", {d, d});
    const HostTensor* wk = need(a + "linear_k.weight", {d, d});
    const HostTensor* wv = need(a + "linear_v.weight", {d, d});
    const HostTensor* bq = need(a + "linear_q.bias", {d});
    const HostTensor* bk = need(a + "linear_k.bias", {d});
    const HostTensor* bv = need(a + "linear_v.bias", {d});
    const HostTensor* wo = need(a + "linear_out.weight", {d, d});
    const HostTensor* bo = need(a + "linear_out.bias", {d});
    const HostTensor* wp = need(a + "linear_pos.weight", {d, d});
    const HostTensor* pu = need(a + "pos_bias_u", {H, dk});
    const HostTensor* pv = need(a + "pos_bias_v", {H, dk});
    if (!missing.empty()) break;
    {
      // fused projection: accumulator columns [q | k | v], each head padded from dk to dkp columns with zero rows;
      // bias = [bq + u | bk | bv], bias2 = bq + v  (multi_head_attention.py:190-193)
      std::vector<float> w(static_cast<size_t>(3) * Dp * d, 0.f), b(3 * Dp, 0.f), b2(Dp, 0.f);
      std::vector<float> wo_p(static_cast<size_t>(d) * Dp, 0.f);
      for (int hh = 0; hh < H; ++hh)
        for (int c = 0; c < dk; ++c) {
          const int src = hh * dk + c, dst = hh * dkp + c;
          memcpy(&w[static_cast<size_t>(dst) * d], &wq->data[static_cast<size_t>(src) * d], d * 4);
          memcpy(&w[static_cast<size_t>(Dp + dst) * d], &wk->data[static_cast<size_t>(src) * d], d * 4);
          memcpy(&w[static_cast<size_t>(2 * Dp + dst) * d], &wv->data[static_cast<size_t>(src) * d], d * 4);
          b[dst] = bq->data[src] + pu->data[src];
          b2[dst] = bq->data[src] + pv->data[src];
          b[Dp + dst] = bk->data[src];
          b[2 * Dp + dst] = bv->data[src];
          memcpy(&wpos[(static_cast<size_t>(l) * Dp + dst) * d], &wp->data[static_cast<size_t>(src) * d], d * 4);
          for (int n = 0; n < d; ++n) wo_p[static_cast<size_t>(n) * Dp + dst] = wo->data[static_cast<size_t>(n) * d + src];
        }
      lw.w_qkv = ab.put_mat(w, f32);
      lw.b_qkv = ab.put_f32(b);
      lw.b_qv = ab.put_f32(b2);
      lw.w_out = ab.put_mat(wo_p, f32);
      lw.b_out = ab.put_f32(bo->data);
    }
    const std::string c = p + "conv.";
    const HostTensor* p1w = need(c + "pointwise_conv1.weight", {2 * d, d, 1});
    const HostTensor* p1b = need(c + "pointwise_conv1.bias", {2 * d});
    const HostTensor* dww = need(c + "depthwise_conv.weight", {d, 1, ks});
    const HostTensor* dwb = need(c + "depthwise_conv.bias", {d});
    const HostTensor* bng = need(c + "batch_norm.weight", {d});
    const HostTensor* bnb = need(c + "batch_norm.bias", {d});
    const HostTensor* bnm = need(c + "batch_norm.running_mean", {d});
    const HostTensor* bnv = need(c + "batch_norm.running_var", {d});
    const HostTensor* p2w = need(c + "pointwise_conv2.weight", {d, d, 1});
    const HostTensor* p2b = need(c + "pointwise_conv2.bias", {d});
    if (!missing.empty()) break;
    {
      // GLU interleave: accumulator columns in groups of 32 = [16 value channels | their 16 gate channels]
      std::vector<float> w(static_cast<size_t>(2) * d * d), b(2 * d);
      for (int col = 0; col < 2 * d; ++col) {
        const int grp = col / 32, j = col % 32;
        const int src = (j < 16) ? grp * 16 + j : d + grp * 16 + (j - 16);
        memcpy(&w[static_cast<size_t>(col) * d], &p1w->data[static_cast<size_t>(src) * d], d * 4);
        b[col] = p1b->data[src];
      }
      lw.w_pw1 = ab.put_mat(w, f32);
      lw.b_pw1 = ab.put_f32(b);
      // eval BatchNorm folded into the depth-wise taps (conformer_modules.py:168-175)
      std::vector<float> taps(static_cast<size_t>(d) * ks), bias(d);
      for (int ch = 0; ch < d; ++ch) {
        const double s = static_cast<double>(bng->data[ch]) / sqrt(static_cast<double>(bnv->data[ch]) + 1e-5);
        for (int k = 0; k < ks; ++k) taps[static_cast<size_t>(k) * d + ch] = static_cast<float>(dww->data[ch * ks + k] * s);  // tap-major
        bias[ch] = static_cast<float>((static_cast<double>(dwb->data[ch]) - bnm->data[ch]) * s + bnb->data[ch]);
      }
      lw.dw_taps = ab.put_f32(taps);
      lw.dw_bias = ab.put_f32(bias);
      {
        // (32, d) block for the fused depthwise + pointwise_conv2 kernel (conv_tail.cu): 31 centred taps + the bias row
        std::vector<float> t32(static_cast<size_t>(32) * d, 0.f);
        const int shift = 15 - (ks - 1) / 2;
        for (int k = 0; k < ks; ++k) memcpy(&t32[static_cast<size_t>(k + shift) * d], &taps[static_cast<size_t>(k) * d], d * 4);
        memcpy(&t32[static_cast<size_t>(31) * d], bias.data(), d * 4);
        lw.dw_taps32 = ab.put_f32(t32);
      }
      lw.w_pw2 = ab.put_mat(p2w->data, f32);
      lw.b_pw2 = ab.put_f32(p2b->data);
    }
  }
  if (!missing.empty()) return fail(h, CFB_ERR_MISSING_WEIGHT, "cfb_finalize_weights: " + missing);
  h->w_pos = ab.put_mat(wpos, f32);
  if (h->has_out_proj) {
    const HostTensor* w = need("out_proj.weight", {h->d_out, d});
    const HostTensor* b = need("out_proj.bias", {h->d_out});
    if (!missing.empty()) return fail(h, CFB_ERR_MISSING_WEIGHT, "cfb_finalize_weights: " + missing);
    h->w_oproj = ab.put_mat(w->data, f32);
    h->b_oproj = ab.put_f32(b->data);
  }

  cudaSetDevice(h->device);
  if (h->arena) cudaFree(h->arena);
  h->arena = nullptr;
  h->arena_bytes = align_up(ab.img.size());
  cudaError_t e = cudaMalloc(&h->arena, h->arena_bytes);
  if (e == cudaSuccess) e = cudaMemcpy(h->arena, ab.img.data(), ab.img.size(), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return fail(h, CFB_ERR_CUDA, std::string("cfb_finalize_weights: ") + cudaGetErrorString(e));
  h->staged.clear();
  h->finalized = true;
  return CFB_OK;
}

int cfb_output_frames(const cfb_handle* h, int T, int* t_out) {
  if (!h || !t_out || T < 1) return fail(h, CFB_ERR_INVALID_ARG, "cfb_output_frames: bad argument");
  *t_out = conv_out(conv_out(T));
  return CFB_OK;
}

int cfb_workspace_bytes(const cfb_handle* h, int B, int T, size_t* out) {
  if (!h || !out || B < 1 || T < 1) return fail(h, CFB_ERR_INVALID_ARG, "cfb_workspace_bytes: bad argument");
  *out = dense_workspace(h, B, T);
  return CFB_OK;
}

int cfb_last_launch_count(const cfb_handle* h) { return h ? h->launches : 0; }

int cfb_set_profiling(cfb_handle* h, int on) {
  if (!h) return CFB_ERR_INVALID_ARG;
  cudaSetDevice(h->device);
  if (on && h->ev_pool.empty()) {
    h->ev_pool.resize(16384);
    for (auto& e : h->ev_pool)
      if (cudaEventCreate(&e) != cudaSuccess) return fail(h, CFB_ERR_CUDA, "cfb_set_profiling: cudaEventCreate failed");
  }
  h->profiling = on != 0;
  h->ev_used = 0;
  h->recs.clear();
  return CFB_OK;
}

int cfb_profile_report(cfb_handle* h, char* buf, size_t cap) {
  if (!h || !buf || cap == 0) return CFB_ERR_INVALID_ARG;
  std::map<std::string, std::pair<int, double>> agg;
  std::vector<std::string> order;
  for (const auto& r : h->recs) {
    cudaEventSynchronize(h->ev_pool[r.e1]);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev_pool[r.e0], h->ev_pool[r.e1]) != cudaSuccess) continue;
    auto it = agg.find(r.label);
    if (it == agg.end()) {
      order.push_back(r.label);
      agg[r.label] = {1, ms};
    } else {
      it->second.first += 1;
      it->second.second += ms;
    }
  }
  std::string out;
  for (const auto& k : order) {
    char line[256];
    snprintf(line, sizeof(line), "%s\t%d\t%.6f\n", k.c_str(), agg[k].first, agg[k].second);
    out += line;
  }
  snprintf(buf, cap, "%s", out.c_str());
  h->ev_used = 0;
  h->recs.clear();
  return CFB_OK;
}

int cfb_debug_buffer(const cfb_handle* h, int B, int T, const char* name, size_t* offset, size_t* bytes) {
  if (!h || !name || !offset || !bytes || B < 1 || T < 1) return fail(h, CFB_ERR_INVALID_ARG, "cfb_debug_buffer: bad argument");
  if (dense_parts(h, B) > 1)
    return fail(h, CFB_ERR_INVALID_ARG, "cfb_debug_buffer: a bf16 batch of B >= 8 runs as two half-batches, each with a "
                                        "workspace plan of its own; ask for B <= 7, or use fp32_validate");
  static const struct {
    const char* name;
    Region Plan::*region;
  } named[] = {{"y1", &Plan::y1},   {"y2", &Plan::y2}, {"x", &Plan::x}, {"a", &Plan::a},   {"h", &Plan::hbuf},
               {"qkv", &Plan::qkv}, {"ctx", &Plan::ctx}, {"g", &Plan::g}, {"c", &Plan::c}, {"pe", &Plan::pe},
               {"pos", &Plan::pos}};
  const Plan p = make_plan(h, B, T);
  for (const auto& n : named)
    if (strcmp(name, n.name) == 0) {
      *offset = (p.*n.region).off;
      *bytes = (p.*n.region).bytes;
      return CFB_OK;
    }
  return fail(h, CFB_ERR_INVALID_ARG, std::string("cfb_debug_buffer: unknown buffer ") + name);
}

}  // extern "C"

namespace {

// Enqueues the launch groups of one forward call.  Each group gets an NVTX range named like its label in the profile
// report (nsys / ncu --nvtx group kernels by them) and, while profiling is on, a CUDA event on either side; its kernels
// are added to the call's launch count, and its failure becomes the handle's error text.  After a failure nothing more
// is enqueued: every later group returns the same status, which the call returns.
struct Enqueue {
  cfb_handle* h;
  unsigned int ev_flags = cudaEventRecordDefault;
  int rc = CFB_OK;
  std::string err;  // a launcher's own description of its failure

  Enqueue(cfb_handle* h_, cudaStream_t st) : h(h_) {
    h->launches = 0;
    if (!h->profiling) return;
    // A profiled forward runs on the caller's stream alone.  Under stream capture the brackets become event-record NODES
    // of the graph (cudaEventRecordExternal): every replay re-records them on the GPU's own timeline, so the intervals
    // hold the kernel and the node-to-node launch latency the replayed step really pays, but none of the host's enqueue
    // cost (eager brackets around a 5 us kernel measure mostly how fast the host enqueues: the GPU runs ahead of it).
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive) ev_flags = cudaEventRecordExternal;
    // calibration of the brackets themselves: two event records with nothing between them (a bracket around a kernel
    // holds the same fixed cost on top of the kernel's launch latency and run time)
    (*this)(st, "(empty bracket)", 0, [] { return 0; });
  }

  // launch() enqueues n kernels on st and returns 0 or an error code
  template <typename Launch>
  int operator()(cudaStream_t st, const char* label, int n, Launch&& launch) {
    if (rc != CFB_OK) return rc;
    nvtxRangePushA(label);
    const bool timed = h->profiling && h->ev_used + 2 <= h->ev_pool.size();
    const size_t e0 = h->ev_used;
    if (timed) cudaEventRecordWithFlags(h->ev_pool[e0], st, ev_flags);
    const int r = launch();
    nvtxRangePop();
    if (timed) {
      cudaEventRecordWithFlags(h->ev_pool[e0 + 1], st, ev_flags);
      h->recs.push_back({label, e0, e0 + 1});
      h->ev_used += 2;
    }
    if (r != 0)
      return rc = fail(h, CFB_ERR_CUDA, std::string("cfb_forward: ") + label + " failed: " +
                                           (err.empty() ? cudaGetErrorString(static_cast<cudaError_t>(r)) : err));
    h->launches += n;
    return CFB_OK;
  }
};

// Runs a batch as n parts: part 0 on the caller's stream st, part g on group_stream[g], forked from st with one event
// and joined back into it (capturable).  part(g, stream) enqueues part g and returns its status.  The parts' kernels
// interleave on the GPU: one part's memory-bound kernels and kernel tails overlap another part's GEMMs.  The join
// happens even after an error, so that a capture in progress is not left with a dangling branch.
template <typename Part>
int run_parts(cfb_handle* h, cudaStream_t st, int n, Part&& part) {
  if (n == 1) return part(0, st);
  int forked = 1;  // streams waiting on the fork, st included
  if (cudaEventRecord(h->ev_fork, st) == cudaSuccess)
    while (forked < n && cudaStreamWaitEvent(h->group_stream[forked], h->ev_fork, 0) == cudaSuccess) ++forked;
  int rc = forked == n ? CFB_OK : fail(h, CFB_ERR_CUDA, "cfb_forward: stream fork failed");
  for (int g = 0; g < n && rc == CFB_OK; ++g) rc = part(g, g == 0 ? st : h->group_stream[g]);
  for (int g = 1; g < forked; ++g) {
    cudaEventRecord(h->group_join[g], h->group_stream[g]);
    cudaStreamWaitEvent(st, h->group_join[g], 0);
  }
  return rc;
}

// Whether a forward runs the conv-module tail as one kernel (conv_tail.cu) instead of two.  CFB_FUSED_TAIL=0 keeps the
// two launches, =2 fuses whenever the shape allows, unset leaves it to the heuristic; it is read on every call (tests
// switch it between forwards).  The fused kernel runs one CTA per 128 frames of a sequence: worth it when the `ctas` of
// the whole batch (its parts run concurrently) fill most of the machine; a CTA takes ~29 us however few there are
// (measured r02f: 128 CTAs 29 us vs 39 us for the two kernels, 59 CTAs 29 us vs 25 us).
bool use_fused_tail(const cfb_handle* h, long long ctas) {
  const char* var = getenv("CFB_FUSED_TAIL");
  const int mode = var != nullptr ? atoi(var) : 1;
  if (mode == 0 || h->validate || !dw_pw_supported(h->d)) return false;
  if (mode == 2) return true;
  const long long waves = (ctas + h->sms - 1) / h->sms;
  return ctas * 100 >= waves * h->sms * 65;
}

// The checks cfb_forward and cfb_forward_packed (`fn` in the messages) share.
int check_forward(cfb_handle* h, const char* fn, const void* feats, int feats_dtype, const void* encoded, int out_dtype,
                  const int32_t* encoded_len, const void* workspace, int B, int T) {
  if (!h) return CFB_ERR_INVALID_ARG;
  auto bad = [&](int code, const char* msg) { return fail(h, code, std::string(fn) + msg); };
  if (!h->finalized) return bad(CFB_ERR_STATE, ": weights are not finalized");
  if (!feats || !encoded || !encoded_len || !workspace || B < 1 || T < 1) return bad(CFB_ERR_INVALID_ARG, ": null pointer or empty batch");
  if (feats_dtype != CFB_F32 && feats_dtype != CFB_BF16) return bad(CFB_ERR_INVALID_ARG, ": feats must be f32 or bf16");
  if (out_dtype != CFB_F32 && out_dtype != CFB_BF16) return bad(CFB_ERR_INVALID_ARG, ": encoded must be f32 or bf16");
  return CFB_OK;
}

// One part of a batch on stream st, in the workspace ws laid out by pl: a contiguous range of B utterances (the whole
// batch, or one half of it), or with pk a group of the B utterances in the packed layout (every utterance in its own slot
// of token rows, no padding; cfb_forward_packed has computed encoded_len and cleared the result).
int forward_range(cfb_handle* h, Enqueue& q, cudaStream_t st, const Plan& pl, const PackedShape* pk, bool fused_tail,
                  const void* feats, int feats_dtype, const int64_t* lengths, int B, int T, void* encoded, int out_dtype,
                  int32_t* encoded_len, uint8_t* ws) {
  const int Bk = pk ? 1 : B;  // batch extent the kernels see: a packed batch is one long sequence
  const bool v = h->validate;
  const bool abf = !v;  // activations / matrices in bf16
  const int d = h->d, C = h->C, F2 = h->F2, dff = h->dff, H = h->H, Dp = h->Dp, L = h->L;
  const int N = pl.N, T2 = pl.T2;
  PackedTables tb;
  if (pk) tb = carve_tables(ws + pl.tables.off, pk->count, pk->n_rows);
  float* raw = v ? reinterpret_cast<float*>(ws + pl.raw.off) : nullptr;

  // one launch on the tensor cores, two on the fp32 validation path
  auto gemm = [&](const void* A, long long lda, const Slot& W, long long ldw, int M, int Nn, int K, int epi, bool out_bf16,
                  EpiParams ep, const char* label) {
    GemmDesc g;
    g.A = A;
    g.lda = lda;
    g.W = h->arena + W.off;
    g.ldw = ldw;
    g.M = M;
    g.N = Nn;
    g.K = K;
    g.epi = epi;
    g.out_bf16 = out_bf16;
    g.ep = ep;
    return q(st, label, v ? 2 : 1, [&] { return v ? launch_gemm_simt(g, raw, st, &q.err) : launch_gemm_tc(g, st, &q.err); });
  };

  // ---- lengths (subsampling.py:164-171)
  if (pk) {
    q(st, "packed layout tables", 1, [&] {
      return launch_packed_plan(reinterpret_cast<const long long*>(lengths), pk->count, pk->first, pk->step, T, pk->t2_max,
                                pk->n_rows, pk->n_tiles, tb, st);
    });
  } else {
    q(st, "lengths", 1, [&] { return launch_lengths(reinterpret_cast<const long long*>(lengths), encoded_len, B, T, 2, st); });
  }
  // ---- subsampling: conv 1->C, conv C->C, linear (subsampling.py:172-175)
  // bf16 path: patch gather + tcgen05 GEMM (the same form dense and packed, so the two stay bit-identical); the CUDA-core
  // kernel below serves the fp32 validation path
  if (pk || !v) {
    q(st, "subsample conv 0 (gather)", 1, [&] {
      return pk ? launch_conv0_im2col_packed(feats, feats_dtype == CFB_BF16, reinterpret_cast<const long long*>(lengths),
                                             ws + pl.a0.off, pk->first, pk->step, h->F0, T, conv_out(T), h->F1, h->Fh,
                                             pk->n_rows, tb, st)
                : launch_conv0_im2col(feats, feats_dtype == CFB_BF16, ws + pl.a0.off, B, h->F0, T, pl.T1, h->F1, pl.Th,
                                      h->Fh, st);
    });
    EpiParams ep;
    ep.out = ws + pl.y1.off;
    ep.ldo = C;
    gemm(ws + pl.a0.off, kConv0Cols, h->sub_w1g, kConv0Cols, Bk * 4 * pl.Th * h->Fh, C, kConv0Cols, EPI_RELU, true, ep,
         "subsample conv 0");
  } else {
    q(st, "subsample conv 0", 1, [&] {
      return launch_subsample_first(feats, feats_dtype == CFB_BF16, h->at<float>(h->sub_w1), h->at<float>(h->sub_b1),
                                    ws + pl.y1.off, abf, B, h->F0, T, C, pl.T1, h->F1, pl.Th, h->Fh, st);
    });
  }
  if (v) {
    q(st, "im2col", 1, [&] {
      return launch_im2col(reinterpret_cast<const float*>(ws + pl.y1.off), reinterpret_cast<float*>(ws + pl.cols.off), B, C,
                           pl.Th, h->Fh, T2, F2, st);
    });
    EpiParams ep;
    ep.bias = h->at<float>(h->sub_b2);
    ep.out = ws + pl.y2.off;
    ep.ldo = C;
    gemm(ws + pl.cols.off, 9LL * C, h->sub_w2, 9LL * C, N * F2, C, 9 * C, EPI_RELU, false, ep, "subsample conv 2");
  } else {
    ConvDesc cd;
    cd.y_in = ws + pl.y1.off;
    cd.W = h->arena + h->sub_w2.off;
    cd.bias = h->at<float>(h->sub_b2);
    cd.y_out = ws + pl.y2.off;
    cd.B = Bk;
    cd.C_in = C;
    cd.C_out = C;
    cd.Th = pl.Th;
    cd.Fh = h->Fh;
    cd.To = T2;
    cd.Fo = F2;
    q(st, "subsample conv 2", 1, [&] { return launch_conv_tc(cd, st, &q.err); });
  }
  float* x = reinterpret_cast<float*>(ws + pl.x.off);
  {
    EpiParams ep;
    ep.bias = h->at<float>(h->sub_b3);
    ep.out = x;
    ep.ldo = d;
    gemm(ws + pl.y2.off, static_cast<long long>(F2) * C, h->sub_w3, static_cast<long long>(F2) * C, N, d, F2 * C, EPI_LINEAR,
         false, ep, "pre_encode.out");
  }
  // ---- relative positional table and its per-layer projections (multi_head_attention.py:186-188, 296-316)
  const int T2pos = pk ? pk->t2_max : T2;  // extent of the relative-position table
  q(st, "pos table", 1, [&] { return launch_pos_table(ws + pl.pe.off, abf, h->at<float>(h->div_term), T2pos, d, st); });
  {
    EpiParams ep;
    ep.out = ws + pl.pos.off;
    ep.ldo = static_cast<long long>(L) * Dp;
    gemm(ws + pl.pe.off, d, h->w_pos, d, pl.P, L * Dp, d, EPI_LINEAR, abf, ep, "linear_pos");
  }
  if (abf) {
    // the attention kernels compute the position term from fp16 operands into an fp16 accumulator (attention_tc.cu): the
    // projections of all layers are converted once, in place
    q(st, "linear_pos -> fp16", 1, [&] {
      return launch_bf16_to_f16(ws + pl.pos.off, static_cast<long long>(L) * Dp, ws + pl.pos.off, pl.P, L * Dp, st);
    });
  }

  const int32_t* lens = encoded_len;
  void* a = ws + pl.a.off;
  for (int l = 0; l < L; ++l) {
    const LayerW& lw = h->layers[l];
    // -- feed forward 1 (conformer_modules.py:98-101)
    for (int f = 0; f < 2; ++f) {
      if (f == 1) {
        // -- self attention (conformer_modules.py:103-110)
        q(st, "norm_self_att", 1, [&] {
          return launch_layernorm(x, h->at<float>(lw.ln_g[1]), h->at<float>(lw.ln_b[1]), a, abf, N, d, nullptr, 1, st);
        });
        EpiParams ep;
        ep.bias = h->at<float>(lw.b_qkv);
        ep.bias2 = h->at<float>(lw.b_qv);
        ep.out = ws + pl.qkv.off;
        ep.ldo = 4LL * Dp;
        ep.qkv_dp = Dp;
        gemm(a, d, lw.w_qkv, d, N, 3 * Dp, d, EPI_QKV, abf, ep, "qkv projection");
        AttnDesc ad;
        ad.qkv = ws + pl.qkv.off;
        ad.pos = ws + pl.pos.off + static_cast<size_t>(l) * Dp * h->esz();
        ad.ld_pos = static_cast<long long>(L) * Dp;
        ad.pos_f16 = abf;
        ad.ctx = ws + pl.ctx.off;
        ad.lens = lens;
        ad.B = B;
        ad.T = T2pos;
        ad.H = H;
        ad.dk = h->dk;
        ad.dkp = h->dkp;
        if (pk) {
          ad.tiles = tb.tiles;
          ad.n_tiles = pk->n_tiles;
          ad.rows = N;
        }
        q(st, "rel-pos attention", 1, [&] { return v ? launch_attn_simt(ad, st, &q.err) : launch_attn_tc(ad, st, &q.err); });
        EpiParams eo;
        eo.bias = h->at<float>(lw.b_out);
        eo.out = x;
        eo.ldo = d;
        eo.alpha = 1.f;
        gemm(ws + pl.ctx.off, Dp, lw.w_out, Dp, N, d, Dp, EPI_RESID, false, eo, "linear_out");
        // -- convolution module (conformer_modules.py:112-114, 160-180)
        q(st, "norm_conv", 1, [&] {
          return launch_layernorm(x, h->at<float>(lw.ln_g[2]), h->at<float>(lw.ln_b[2]), a, abf, N, d, nullptr, 1, st);
        });
        EpiParams eg;
        eg.bias = h->at<float>(lw.b_pw1);
        eg.out = ws + pl.g.off;
        eg.ldo = d;
        if (pk) {
          eg.row_t = tb.row_t;  // zero at the gap rows: the depth-wise halo of a slot must not see its neighbours
        } else {
          eg.lens = lens;
          eg.frames_per_seq = T2;
        }
        gemm(a, d, lw.w_pw1, d, N, 2 * d, d, EPI_GLU, abf, eg, "pointwise_conv1+glu");
        if (fused_tail) {
          // depthwise + BatchNorm + Swish + pointwise_conv2 + residual in one kernel (conv_tail.cu)
          DwPwDesc dp;
          dp.g = ws + pl.g.off;
          dp.taps32 = h->at<float>(lw.dw_taps32);
          dp.W = h->arena + lw.w_pw2.off;
          dp.bias2 = h->at<float>(lw.b_pw2);
          dp.x = x;
          dp.B = Bk;
          dp.T = T2;
          dp.d = d;
          q(st, "depthwise+pointwise_conv2", 1, [&] { return launch_dw_pw(dp, st, &q.err); });
        } else {
          q(st, "depthwise conv", 1, [&] {
            return launch_depthwise(ws + pl.g.off, h->at<float>(lw.dw_taps), h->at<float>(lw.dw_bias), ws + pl.c.off, abf, Bk,
                                    T2, d, h->ksize, st);
          });
          EpiParams e2;
          e2.bias = h->at<float>(lw.b_pw2);
          e2.out = x;
          e2.ldo = d;
          e2.alpha = 1.f;
          gemm(ws + pl.c.off, d, lw.w_pw2, d, N, d, d, EPI_RESID, false, e2, "pointwise_conv2");
        }
      }
      const int ln = f == 0 ? 0 : 3;
      if (!(f == 0 && l > 0 && abf)) {  // bf16 path: norm_feed_forward1 of layers > 0 is fused into the previous norm_out
        q(st, "norm_feed_forward", 1, [&] {
          return launch_layernorm(x, h->at<float>(lw.ln_g[ln]), h->at<float>(lw.ln_b[ln]), a, abf, N, d, nullptr, 1, st);
        });
      }
      EpiParams e1;
      e1.bias = h->at<float>(lw.ff_b1[f]);
      e1.out = ws + pl.hbuf.off;
      e1.ldo = dff;
      gemm(a, d, lw.ff_w1[f], d, N, dff, d, EPI_SWISH, abf, e1, "linear1+swish");
      EpiParams e2;
      e2.bias = h->at<float>(lw.ff_b2[f]);
      e2.out = x;
      e2.ldo = d;
      e2.alpha = 0.5f;  // fc_factor (conformer_modules.py:57,101,118)
      gemm(ws + pl.hbuf.off, dff, lw.ff_w2[f], dff, N, d, dff, EPI_RESID, false, e2, "linear2");
    }
    // -- norm_out (conformer_modules.py:120); the last one writes the result
    const bool last = l == L - 1;
    const float* g4 = h->at<float>(lw.ln_g[4]);
    const float* b4 = h->at<float>(lw.ln_b[4]);
    q(st, "norm_out", 1, [&] {
      if (last && pk)  // the valid rows of every slot into the dense (B, T', d) result of the reference API (packed.cu)
        return launch_layernorm_scatter(x, g4, b4, encoded, out_dtype == CFB_BF16, N, d, tb.row_out, st);
      if (last && !h->has_out_proj) return launch_layernorm(x, g4, b4, encoded, out_dtype == CFB_BF16, N, d, lens, T2, st);
      if (last) return launch_layernorm(x, g4, b4, a, abf, N, d, nullptr, 1, st);
      if (abf) {
        const LayerW& nx = h->layers[l + 1];
        return launch_layernorm_dual(x, g4, b4, x, h->at<float>(nx.ln_g[0]), h->at<float>(nx.ln_b[0]), a, N, d, st);
      }
      return launch_layernorm(x, g4, b4, x, false, N, d, nullptr, 1, st);
    });
  }
  if (h->has_out_proj) {  // conformer_encoder.py:277-278
    EpiParams ep;
    ep.bias = h->at<float>(h->b_oproj);
    ep.out = encoded;
    ep.ldo = h->d_out;
    ep.lens = lens;
    ep.frames_per_seq = T2;
    gemm(a, d, h->w_oproj, d, N, h->d_out, d, EPI_LINEAR, out_dtype == CFB_BF16, ep, "out_proj");
  }
  return q.rc;
}

}  // namespace

extern "C" {

int cfb_forward(cfb_handle* h, const void* feats, int feats_dtype, const int64_t* lengths, int B, int T, void* encoded,
                int out_dtype, int32_t* encoded_len, void* workspace, size_t ws_bytes, cfb_stream stream) {
  if (int rc = check_forward(h, "cfb_forward", feats, feats_dtype, encoded, out_dtype, encoded_len, workspace, B, T)) return rc;
  if (ws_bytes < dense_workspace(h, B, T) || (reinterpret_cast<uintptr_t>(workspace) & 255))
    return fail(h, CFB_ERR_WORKSPACE, "cfb_forward: workspace too small or not 256-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int t_out = conv_out(conv_out(T));
  set_pdl_auto(static_cast<long long>(B) * t_out <= 4096);
  const bool fused_tail = use_fused_tail(h, static_cast<long long>(B) * ((t_out + 127) / 128));
  Enqueue q(h, st);
  // Utterances are independent, so a batch can run as two half-batches on two streams (run_parts).  Results are
  // identical to the single-stream schedule (every row sees the same padded extent T).  Off while per-kernel profiling
  // is on.
  const int n = h->profiling ? 1 : dense_parts(h, B);
  const size_t in_es = feats_dtype == CFB_F32 ? 4 : 2, out_es = out_dtype == CFB_F32 ? 4 : 2;
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  return run_parts(h, st, n, [&](int i, cudaStream_t s) {
    const Range r = dense_part(B, n, i);
    const Plan pl = make_plan(h, r.count, T);
    const int rc = forward_range(h, q, s, pl, nullptr, fused_tail,
                                 reinterpret_cast<const uint8_t*>(feats) + static_cast<size_t>(r.first) * h->F0 * T * in_es,
                                 feats_dtype, lengths ? lengths + r.first : nullptr, r.count, T,
                                 reinterpret_cast<uint8_t*>(encoded) + static_cast<size_t>(r.first) * t_out * h->d_out * out_es,
                                 out_dtype, encoded_len + r.first, ws);
    ws += pl.total;
    return rc;
  });
}

}  // extern "C"

// A small packed batch runs as interleaved groups (utterances g, g + G, ...: balanced when the caller sorts by length,
// as sharding.plan_shards does) on their own streams, like cfb_forward's half-batches: the groups' kernels
// interleave on the GPU, which matters most for SMALL shares (a rank of an 8-GPU job), where every kernel is a fraction
// of a wave and latency-bound.
// Measured (r5b / r5e, cfg3 shares, ms per step): 25 480 rows 13.31 with two groups / 13.25 with one, 6 500 rows 4.41 /
// 4.17, 3 100 rows (an 8-GPU share) 2.80 with one or two groups, 2.73 with three -- it only pays once a launch no
// longer fills the machine.
constexpr int kSmallBatchRows = 4096;
// number of interleaved groups a packed batch runs as (1 = no split)
static int packed_groups(const cfb_handle* h, int B, int n_rows) {
  const char* force = getenv("CFB_PACKED_GROUPS");  // 1 .. 4 forces (read per call: tests switch it)
  int g = 1;
  if (force != nullptr) g = atoi(force);
  else if (n_rows <= kSmallBatchRows) g = 3;  // r5e: 1 / 2 / 3 / 4 groups 2.80 / 2.81 / 2.73 / 2.75 ms
  if (h->profiling) g = 1;
  g = std::min(std::min(g, B), cfb_handle::kMaxGroups);
  return std::max(g, 1);
}

extern "C" {

int cfb_packed_workspace_bytes(const cfb_handle* h, const int64_t* lengths_host, int B, int T, size_t* out) {
  if (!h || !out || B < 1 || T < 1) return fail(h, CFB_ERR_INVALID_ARG, "cfb_packed_workspace_bytes: bad argument");
  *out = packed_workspace(h, lengths_host, B, T);
  return CFB_OK;
}

int cfb_forward_packed(cfb_handle* h, const void* feats, int feats_dtype, const int64_t* lengths, const int64_t* lengths_host,
                       int B, int T, void* encoded, int out_dtype, int32_t* encoded_len, void* workspace, size_t ws_bytes,
                       cfb_stream stream) {
  if (int rc = check_forward(h, "cfb_forward_packed", feats, feats_dtype, encoded, out_dtype, encoded_len, workspace, B, T))
    return rc;
  if ((lengths == nullptr) != (lengths_host == nullptr))
    return fail(h, CFB_ERR_INVALID_ARG, "cfb_forward_packed: lengths and lengths_host must both be given (or both NULL)");
  if (h->validate) return fail(h, CFB_ERR_UNSUPPORTED, "cfb_forward_packed: the fp32 validation path runs dense batches only");
  if (h->has_out_proj) return fail(h, CFB_ERR_UNSUPPORTED, "cfb_forward_packed: out_proj (feat_out != d_model) runs dense batches only");
  if (B > 2048) return fail(h, CFB_ERR_UNSUPPORTED, "cfb_forward_packed: at most 2048 utterances per call");
  if (ws_bytes < packed_workspace(h, lengths_host, B, T) || (reinterpret_cast<uintptr_t>(workspace) & 255))
    return fail(h, CFB_ERR_WORKSPACE, "cfb_forward_packed: workspace too small or not 256-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const PackedShape ps = packed_shape(lengths_host, B, T);
  set_pdl_auto(ps.n_rows <= kSmallBatchRows);
  const bool fused_tail = use_fused_tail(h, (ps.n_rows + 127) / 128);
  const int n = packed_groups(h, B, ps.n_rows);
  Enqueue q(h, st);
  // encoded_len and the cleared dense result are needed by every group: enqueue them, then fork
  if (q(st, "lengths", 1, [&] { return launch_lengths(reinterpret_cast<const long long*>(lengths), encoded_len, B, T, 2, st); }))
    return q.rc;
  const size_t out_bytes = static_cast<size_t>(B) * ps.t2_max * h->d * (out_dtype == CFB_BF16 ? 2 : 4);
  if (cudaMemsetAsync(encoded, 0, out_bytes, st) != cudaSuccess) return fail(h, CFB_ERR_CUDA, "cfb_forward_packed: memset failed");
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  return run_parts(h, st, n, [&](int g, cudaStream_t s) {
    const PackedShape gs = packed_shape(lengths_host, B, T, g, n);
    const Plan pl = make_plan(h, B, T, &gs);
    const int rc = forward_range(h, q, s, pl, &gs, fused_tail, feats, feats_dtype, lengths, B, T, encoded, out_dtype,
                                 encoded_len, ws);
    ws += pl.total;
    return rc;
  });
}

// ---------------------------------------------------------------------------------------------------------------------
// kernel-level entry points
namespace {
std::string g_op_error;
int op_fail(int rc, const std::string& err) {
  g_op_error = err.empty() ? std::string(cudaGetErrorString((cudaError_t)rc)) : err;
  g_create_error = g_op_error;  // cfb_last_error(NULL) reports handle-less failures
  return CFB_ERR_CUDA;
}
int op_refuse(int code, const std::string& err) {
  g_op_error = err;
  g_create_error = g_op_error;
  return code;
}

// The (epilogue, output type, shape) combinations the GEMM kernels can write; anything else would store another type's
// rows into `out`, write past its rows or read past bias2, so it is refused before anything is enqueued.
int gemm_args_error(int use_tc, int epi, int N, int64_t ldo, int out_dtype, int qkv_dp) {
  if (epi < CFB_EPI_LINEAR || epi > CFB_EPI_GLU) return op_refuse(CFB_ERR_INVALID_ARG, "op_gemm: unknown epilogue");
  if (out_dtype != CFB_F32 && out_dtype != CFB_BF16)
    return op_refuse(CFB_ERR_UNSUPPORTED, "op_gemm: out_dtype must be CFB_F32 or CFB_BF16");
  if (epi == CFB_EPI_RESID && out_dtype != CFB_F32)
    return op_refuse(CFB_ERR_UNSUPPORTED, "op_gemm: the residual epilogue adds into an fp32 stream (out_dtype CFB_F32)");
  if (use_tc && out_dtype == CFB_F32 && epi != CFB_EPI_LINEAR && epi != CFB_EPI_RESID)
    return op_refuse(CFB_ERR_UNSUPPORTED, "op_gemm: on tensor cores only the linear and residual epilogues write fp32");
  if (epi == CFB_EPI_QKV && (qkv_dp <= 0 || qkv_dp % 64 || static_cast<int64_t>(N) != 3 * static_cast<int64_t>(qkv_dp)))
    return op_refuse(CFB_ERR_INVALID_ARG, "op_gemm: QKV needs qkv_dp > 0, qkv_dp % 64 == 0 and N == 3 * qkv_dp");
  if (epi == CFB_EPI_GLU && N % 32)
    return op_refuse(CFB_ERR_INVALID_ARG, "op_gemm: GLU needs N % 32 == 0 (groups of [16 a | 16 gate] columns)");
  const int64_t cols = epi == CFB_EPI_QKV ? static_cast<int64_t>(N) + qkv_dp : epi == CFB_EPI_GLU ? N / 2 : N;
  if (ldo < cols) return op_refuse(CFB_ERR_INVALID_ARG, "op_gemm: ldo is smaller than the output's column count");
  return CFB_OK;
}
}  // namespace

int cfb_op_gemm(int use_tc, int epilogue, const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                const float* bias2, int M, int N, int K, void* out, int64_t ldo, int out_dtype, float alpha,
                const int32_t* lens, int frames_per_seq, int qkv_dp, float* scratch, cfb_stream stream) {
  if (int rc = gemm_args_error(use_tc, epilogue, N, ldo, out_dtype, qkv_dp)) return rc;
  GemmDesc g;
  g.A = A;
  g.lda = lda;
  g.W = W;
  g.ldw = ldw;
  g.M = M;
  g.N = N;
  g.K = K;
  g.epi = epilogue;
  g.out_bf16 = out_dtype == CFB_BF16;
  g.ep.bias = bias;
  g.ep.bias2 = bias2;
  g.ep.out = out;
  g.ep.ldo = ldo;
  g.ep.alpha = alpha;
  g.ep.lens = lens;
  g.ep.frames_per_seq = frames_per_seq > 0 ? frames_per_seq : 1;
  g.ep.qkv_dp = qkv_dp;
  std::string err;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int rc = use_tc ? launch_gemm_tc(g, st, &err) : launch_gemm_simt(g, scratch, st, &err);
  return rc == 0 ? CFB_OK : op_fail(rc, err);
}

int cfb_op_layernorm(const float* x, const float* gamma, const float* beta, void* out, int out_dtype, int rows, int d,
                     const int32_t* lens, int frames_per_seq, cfb_stream stream) {
  int rc = launch_layernorm(x, gamma, beta, out, out_dtype == CFB_BF16, rows, d, lens, frames_per_seq > 0 ? frames_per_seq : 1,
                            reinterpret_cast<cudaStream_t>(stream));
  return rc == 0 ? CFB_OK : op_fail(rc, rc == -1 ? "layernorm: d must be a multiple of 4 and <= 1024" : "");
}

int cfb_op_layernorm_dual(const float* x, const float* g1, const float* b1, float* out1, const float* g2, const float* b2,
                          void* out2_bf16, int rows, int d, cfb_stream stream) {
  int rc = launch_layernorm_dual(x, g1, b1, out1, g2, b2, out2_bf16, rows, d, reinterpret_cast<cudaStream_t>(stream));
  return rc == 0 ? CFB_OK : op_fail(rc, rc == -1 ? "layernorm_dual: d must be a multiple of 4 and <= 1024" : "");
}

int cfb_op_depthwise(const void* x, const float* taps, const float* bias, void* out, int dtype, int B, int T, int d,
                     int ksize, cfb_stream stream) {
  int rc = launch_depthwise(x, taps, bias, out, dtype == CFB_BF16, B, T, d, ksize, reinterpret_cast<cudaStream_t>(stream));
  return rc == 0 ? CFB_OK : op_fail(rc, rc == -1 ? "depthwise: ksize must be odd <= 31 and d even" : "");
}

int cfb_op_dw_pw2(const void* g, const float* taps32, const void* W, const float* bias2, float* x, int B, int T, int d,
                  cfb_stream stream) {
  DwPwDesc c;
  c.g = g;
  c.taps32 = taps32;
  c.W = W;
  c.bias2 = bias2;
  c.x = x;
  c.B = B;
  c.T = T;
  c.d = d;
  std::string err;
  int rc = launch_dw_pw(c, reinterpret_cast<cudaStream_t>(stream), &err);
  return rc == 0 ? CFB_OK : op_fail(rc, err);
}

namespace {
int run_logmel(const float* audio, const int64_t* lengths, int B, int L, const float* window, int win_length, int n_fft,
               int hop, const float* fb, const int32_t* fb_span, int n_mels, float preemph, float log_guard, bool normalize,
               float std_eps, float* features, int T_out, int64_t* seq_len, int32_t* flag, cfb_stream stream) {
  LogMelDesc d;
  d.audio = audio;
  d.lengths = lengths;
  d.B = B;
  d.L = L;
  d.window = window;
  d.win_length = win_length;
  d.n_fft = n_fft;
  d.hop = hop;
  d.fb = fb;
  d.fb_span = fb_span;
  d.n_mels = n_mels;
  d.preemph = preemph;
  d.log_guard = log_guard;
  d.normalize = normalize;
  d.std_eps = std_eps;
  d.features = features;
  d.T_out = T_out;
  d.seq_len = seq_len;
  d.flag = flag;
  if (!audio || !lengths || !window || !fb || !fb_span || !features || !seq_len || (normalize && !flag))
    return op_fail(-1, "logmel: null pointer");
  std::string err;
  int rc = launch_logmel(d, reinterpret_cast<cudaStream_t>(stream), &err);
  return rc == 0 ? CFB_OK : op_fail(rc, err);
}
}  // namespace

int cfb_op_logmel(const float* audio, const int64_t* lengths, int B, int L, const float* window, int win_length, int n_fft,
                  int hop, const float* fb, const int32_t* fb_span, int n_mels, float preemph, float log_guard, float std_eps, float* features,
                  int T_out, int64_t* seq_len, int32_t* flag, cfb_stream stream) {
  return run_logmel(audio, lengths, B, L, window, win_length, n_fft, hop, fb, fb_span, n_mels, preemph, log_guard, true, std_eps,
                    features, T_out, seq_len, flag, stream);
}

int cfb_op_logmel_raw(const float* audio, const int64_t* lengths, int B, int L, const float* window, int win_length, int n_fft,
                      int hop, const float* fb, const int32_t* fb_span, int n_mels, float preemph, float log_guard,
                      float* features, int T_out, int64_t* seq_len, cfb_stream stream) {
  return run_logmel(audio, lengths, B, L, window, win_length, n_fft, hop, fb, fb_span, n_mels, preemph, log_guard, false, 0.f,
                    features, T_out, seq_len, nullptr, stream);
}

int cfb_op_feature_buffers(const float* features, int n_files, int F, int T, const int64_t* seq_len,
                           const int32_t* first_window, int n_windows, int frame_len, int buffer_len, float* out,
                           cfb_stream stream) {
  if (!features || !seq_len || !first_window || !out) return op_fail(-1, "feature_buffers: null pointer");
  std::string err;
  int rc = launch_feature_buffers(features, n_files, F, T, reinterpret_cast<const long long*>(seq_len), first_window,
                                  n_windows, frame_len, buffer_len, out, reinterpret_cast<cudaStream_t>(stream), &err);
  return rc == 0 ? CFB_OK : op_fail(rc, err);
}

int cfb_op_rel_attention(int use_tc, const void* qkv, const void* pos, int64_t ld_pos, void* ctx, const int32_t* lens,
                         int B, int T, int H, int dk, int dkp, cfb_stream stream) {
  AttnDesc a;
  a.qkv = qkv;
  a.pos = pos;
  a.ld_pos = ld_pos;
  a.ctx = ctx;
  a.lens = lens;
  a.B = B;
  a.T = T;
  a.H = H;
  a.dk = dk;
  a.dkp = dkp;
  if (use_tc && ((dkp != 64 && dkp != 128) || dk < 1 || dk > dkp)) {
    op_fail(-1, "rel_attention: the tensor-core path takes dkp 64 or 128 and 1 <= dk <= dkp");
    return CFB_ERR_INVALID_ARG;
  }
  std::string err;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int rc = use_tc ? launch_attn_tc(a, st, &err) : launch_attn_simt(a, st, &err);
  return rc == 0 ? CFB_OK : op_fail(rc, err);
}

int cfb_op_lengths(const int64_t* lengths, int32_t* out, int B, int T_full, int n_stages, cfb_stream stream) {
  int rc = launch_lengths(reinterpret_cast<const long long*>(lengths), out, B, T_full, n_stages,
                          reinterpret_cast<cudaStream_t>(stream));
  return rc == 0 ? CFB_OK : op_fail(rc, "");
}

}  // extern "C"
