// Shared declarations of the cfb CUDA library (internal; the public surface is include/cfb.h).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

namespace cfb {

using bf16 = __nv_bfloat16;

// ---- epilogue selection shared by the tensor-core GEMM and the CUDA-core validation GEMM ---------------------
enum EpiKind : int { EPI_LINEAR = 0, EPI_SWISH = 1, EPI_RELU = 2, EPI_RESID = 3, EPI_QKV = 4, EPI_GLU = 5 };

struct EpiParams {
  const float* bias = nullptr;   // per accumulator column (may be null)
  const float* bias2 = nullptr;  // QKV: bias of the q+v copy
  void* out = nullptr;           // TOut* (RESID: float*, read-modify-write)
  long long ldo = 0;             // elements between output rows
  float alpha = 1.f;             // RESID scale
  const int32_t* lens = nullptr; // GLU / LINEAR: valid frames per sequence (null = no masking)
  int frames_per_seq = 1;
  const int32_t* row_t = nullptr; // packed batches: frame index of every output row, < 0 at gap rows (replaces lens)
  int qkv_dp = 0;                // QKV: H * dk_pad
  int M = 0;                     // valid output rows
  int N = 0;                     // accumulator columns
};

// ---- launch descriptions ---------------------------------------------------------------------------------------
struct GemmDesc {
  // D (M x N) = A (M x K) * W^T (N x K); all row-major with the given leading dimensions (elements)
  const void* A = nullptr;
  long long lda = 0;
  const void* W = nullptr;
  long long ldw = 0;
  int M = 0, N = 0, K = 0;
  int epi = EPI_LINEAR;
  bool out_bf16 = true;
  EpiParams ep;
};

// implicit-GEMM view of the second strided 3x3 convolution of the subsampling stack:
// input y1 in the parity-split channels-last layout [B][4 planes][Th][Fh][C] (plane = (t&1)*2 + (f&1)),
// output y2 [B][To][Fo][C] with relu(bias + conv)
struct ConvDesc {
  const void* y_in = nullptr;
  const void* W = nullptr;  // [C_out][9*C_in], k = (kh*3+kw)*C_in + c
  const float* bias = nullptr;
  void* y_out = nullptr;
  int B = 0, C_in = 0, C_out = 0;
  int Th = 0, Fh = 0;  // plane extents of the input
  int To = 0, Fo = 0;  // output extents
};

struct AttnDesc {
  const void* qkv = nullptr;  // (B*T, 4*Dp)
  const void* pos = nullptr;  // (2T-1, ld_pos), this layer's columns start at pos
  long long ld_pos = 0;
  void* ctx = nullptr;  // (B*T, Dp)
  const int32_t* lens = nullptr;
  int B = 0, T = 0, H = 0, dk = 0, dkp = 0;
  // packed batches (PackedTables): qkv / ctx have `rows` token rows, every sequence owns a slot of them; T stays the
  // extent of the positional table (the longest sequence).  tiles == nullptr: the dense (B, T) layout above.
  bool pos_f16 = false;  // pos already holds fp16 (the engine converts its buffer once per forward); false: bf16
  const int4* tiles = nullptr;  // [n_tiles] (sequence, first query row i0, first token row of the slot, rows in the slot)
  int n_tiles = 0;
  long long rows = 0;
};

// ---- packed (variable-length) batches ---------------------------------------------------------------------------
// Every utterance owns a SLOT of token rows: its T'_b valid frames followed by >= 15 gap rows (slot sizes are multiples
// of 8), slots back to back.  Token-major kernels (LayerNorm, GEMMs) simply run over all rows; the depth-wise
// convolution sees one long sequence whose gap rows are zero in its input (its 15-frame halo never reaches a
// neighbour); attention works per slot; the strided convolutions run over the matching "virtual" time axis (4 input
// frames / 2 first-conv rows per token row).  Tables are built on the device from the lengths (packed.cu).
constexpr int kPackGap = 15;   // >= (31 - 1) / 2: the depth-wise halo
constexpr int kPackAlign = 8;  // slot granularity in token rows (= 16 first-conv rows = one im2col block)
struct PackedTables {
  int32_t* seq_row0 = nullptr;  // [B] first token row of the slot
  int32_t* seq_rows = nullptr;  // [B] token rows in the slot
  int32_t* row_t = nullptr;     // [N] frame index inside the utterance, -1 at gap rows
  int32_t* row_out = nullptr;   // [N] row of the dense (B, T2, d) result, -1 at gap rows
  int32_t* blk_seq = nullptr;   // [N / 8] utterance owning every 8-row block
  int4* tiles = nullptr;        // [n_tiles] attention query tiles (b, i0, row0, rows)
};
inline int packed_slot_rows(int t2) { return (t2 + kPackGap + kPackAlign - 1) / kPackAlign * kPackAlign; }
// Lays out the group of B utterances first, first + step, ... of the batch.  lengths: int64 input frames of the WHOLE
// batch on the device (clipped to [0, T]); T2 = dense output extent; n_rows / n_tiles as computed by the host from the
// same lengths.  One CTA.
int launch_packed_plan(const long long* lengths, int B, int first, int step, int T, int T2, int n_rows, int n_tiles,
                       const PackedTables& tb, cudaStream_t st);
// conv0_im2col for the packed layout: rows of slot k come from feats[first + k step]; first-conv rows t1 > T1_b or >= T1
// are zero
int launch_conv0_im2col_packed(const void* feats, bool feats_bf16, const long long* lengths, void* a0, int first, int step,
                               int F, int T, int T1, int F1, int Fh, int n_rows, const PackedTables& tb, cudaStream_t st);
// LayerNorm whose output rows are scattered through row_map (rows with a negative entry are skipped)
int launch_layernorm_scatter(const float* x, const float* gamma, const float* beta, void* out, bool out_bf16, int rows,
                             int d, const int32_t* row_map, cudaStream_t st);

// ---- programmatic dependent launch (PDL) ------------------------------------------------------------------------
// Every product-path kernel is launched with programmaticStreamSerialization: its CTAs may start (barrier init,
// TMEM allocation, descriptor prefetch) while the previous kernel of the stream drains, and they call pdl_wait()
// before their first global-memory access -- it returns once the previous kernel has completed and flushed.
// pdl_launch_dependents() at the top of a kernel lets the NEXT kernel start the same way.  The forward is a chain
// of ~260 short dependent launches, so this can hide launch latency + prologue per link.  The engine turns it on per
// forward for small batches: see pdl_enabled() for the measurement.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

bool pdl_enabled();
void set_pdl_auto(bool on);  // per host thread: the engine enables PDL for small batches (tmap.cu)
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#endif

// ---- launchers (each returns a cudaError_t-compatible int; 0 = success) ------------------------------------------
int launch_gemm_tc(const GemmDesc& g, cudaStream_t st, std::string* err);
// CTA-pair (cta_group::2) variant for N % 256 == 0 (gemm_tc2.cu); launch_gemm_tc picks it by shape / CFB_GEMM_2CTA
bool gemm_tc2_supported(const GemmDesc& g);
int launch_gemm_tc2(const GemmDesc& g, cudaStream_t st, std::string* err);
int launch_conv_tc(const ConvDesc& c, cudaStream_t st, std::string* err);
int launch_gemm_simt(const GemmDesc& g, float* scratch, cudaStream_t st, std::string* err);
// tensor-core attention: dkp 64 -> attention_tc.cu / attention_tcp.cu, dkp 128 -> attention_tc128.cu
int launch_attn_tc(const AttnDesc& a, cudaStream_t st, std::string* err);
// persistent form (one CTA per SM walks over the (query tile, head, sequence) items; attention_tcp.cu)
int launch_attn_tcp(const AttnDesc& a, cudaStream_t st, std::string* err);
// heads 64 < dk <= 128, padded to 128 columns (attention_tc128.cu); per-item form only
int launch_attn_tc128(const AttnDesc& a, cudaStream_t st, std::string* err);
int launch_attn_simt(const AttnDesc& a, cudaStream_t st, std::string* err);
// fp16 view of the positional projections for the tensor-core attention kernels (attention_tc.cu)
const void* attn_pos_f16(const AttnDesc& a, int Dp, cudaStream_t st);
// bf16 (rows x cols, leading dimension ld) -> fp16 (rows x cols, dense); dst == src with ld == cols converts in place
int launch_bf16_to_f16(const void* src, long long ld, void* dst, long long rows, int cols, cudaStream_t st);

int launch_layernorm(const float* x, const float* gamma, const float* beta, void* out, bool out_bf16, int rows, int d,
                     const int32_t* lens, int frames_per_seq, cudaStream_t st);
// y = LN(x; g1, b1) -> out1 (fp32, may alias x); LN(y; g2, b2) -> out2 (bf16): norm_out + the next layer's first norm
int launch_layernorm_dual(const float* x, const float* g1, const float* b1, float* out1, const float* g2, const float* b2,
                          void* out2_bf16, int rows, int d, cudaStream_t st);
int launch_depthwise(const void* x, const float* taps, const float* bias, void* out, bool is_bf16, int B, int T, int d,
                     int ksize, cudaStream_t st);
int launch_lengths(const long long* lengths, int32_t* out, int B, int T_full, int n_stages, cudaStream_t st);
int launch_pos_table(void* out, bool out_bf16, const float* div_term, int T, int d, cudaStream_t st);
// first strided conv (1 -> C channels) + ReLU from (B, F, T) features into the parity-split channels-last layout
int launch_subsample_first(const void* feats, bool feats_bf16, const float* w9, const float* bias, void* y_out,
                           bool out_bf16, int B, int F, int T, int C, int T1, int F1, int Th, int Fh, cudaStream_t st);
// tensor-core form of the first conv: rows [x_hi(9) | x_lo(9) | 1 | 1 | 0 x 4] (bf16, 24 columns) in y1's row order
constexpr int kConv0Cols = 24;
// The gather kernels of the first conv (subsample_first_kernel, conv0_im2col_kernel, conv0_im2col_packed_kernel) stage
// (F + 2) x 34 fp32 features of a block in shared memory, inside the 48 KB a launch gets without opting in: F <= 359.
constexpr int kMaxFeatIn = 359;
int launch_conv0_im2col(const void* feats, bool feats_bf16, void* a0, int B, int F, int T, int T1, int F1, int Th, int Fh,
                        cudaStream_t st);
// validation path: gather the 3x3/s2 patches of a parity-split tensor into a dense (rows x 9*C) fp32 matrix
int launch_im2col(const float* y_in, float* cols, int B, int C, int Th, int Fh, int To, int Fo, cudaStream_t st);

// TMA descriptor encoder (cuTensorMapEncodeTiled resolved through the runtime; libcuda is not linked)
bool encode_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                      const uint32_t* box, std::string* err);
bool encode_tmap(CUtensorMap* map, const void* base, bool is_f32, int rank, const uint64_t* dims,
                 const uint64_t* strides_bytes, const uint32_t* box, std::string* err);

// same with the shared-memory swizzle chosen by the caller (false = rows land densely, for tiles read by SIMT code)
bool encode_tmap_ex(CUtensorMap* map, const void* base, bool is_f32, int rank, const uint64_t* dims,
                    const uint64_t* strides_bytes, const uint32_t* box, bool swizzle128, std::string* err);

// log-mel front-end (frontend.cu): FilterbankFeatures.forward in eval mode, features.py:358-453
struct LogMelDesc {
  const float* audio = nullptr;   // (B, L) fp32 waveforms, zero after each utterance's length
  const void* lengths = nullptr;  // (B) int64 samples
  int B = 0, L = 0;
  const float* window = nullptr;  // (win_length) fp32
  int win_length = 0, n_fft = 512, hop = 160;
  const float* fb = nullptr;      // (n_mels, n_fft / 2 + 1): the mel filter bank (featurizer.fb)
  const int* fb_span = nullptr;   // (n_mels, 2) int32: first non-zero FFT bin and bin count of every filter
  int n_mels = 0;
  float preemph = 0.97f, log_guard = 5.9604644775390625e-08f, std_eps = 1e-5f;
  float* features = nullptr;      // (B, n_mels, T_out) fp32
  int T_out = 0;                  // >= 1 + L / hop; frames from seq_len on are written as zeros
  void* seq_len = nullptr;        // (B) int64
  int* flag = nullptr;            // set to 1 when some utterance has exactly one frame (the reference raises)
  bool normalize = true;          // false: normalize "None" -- no statistics, no flag (flag may be null)
};
int launch_logmel(const LogMelDesc& d, cudaStream_t st, std::string* err);

// buffered long-audio inference (buffered.cu): the normalised overlapping windows of FeatureFrameBufferer
int launch_feature_buffers(const float* feat, int n_files, int F, int T, const long long* seq_len, const int* first_window,
                           int n_windows, int fl, int W, float* out, cudaStream_t st, std::string* err);

// depth-wise conv (+ folded BatchNorm + Swish) fused into pointwise_conv2 and the residual update (conv_tail.cu):
//   x[b,t,:] += W2 * swish(bias_dw + sum_k taps[k] * g[b, t + k - 15, :]) + bias2
// taps32: (32, d) fp32, rows 0..30 = the 31 taps (shorter kernels centred, zero padded), row 31 = the folded bias
struct DwPwDesc {
  const void* g = nullptr;      // (B*T, d) bf16, GLU output with padded frames zeroed
  const float* taps32 = nullptr;
  const void* W = nullptr;      // (d, d) bf16 pointwise_conv2 weight
  const float* bias2 = nullptr; // (d)
  float* x = nullptr;           // (B*T, d) fp32 residual stream, updated in place
  int B = 0, T = 0, d = 0;
};
bool dw_pw_supported(int d);
int launch_dw_pw(const DwPwDesc& c, cudaStream_t st, std::string* err);

}  // namespace cfb
