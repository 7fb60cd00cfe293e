/*
 * cfb.h -- C ABI of the B200-native Conformer encoder forward ("cfb" = conformer forward, Blackwell).
 *
 * This is the drop-in boundary for
 *     ConformerEncoder.forward(audio_signal, length) -> (encoded, encoded_len)
 *     reference: nemo/collections/asr/modules/conformer_encoder.py:231-281
 * Plain C: pointers, sizes and integers only.  No torch / C++ types cross it, no exception crosses it.
 * Every entry point returns 0 (CFB_OK) or a non-zero cfb_status; cfb_last_error() gives the text.
 *
 * The reference side binds it with ctypes (see INTEGRATION.md); the Python wrapper in
 * conformer-nemo_b200/encoder.py is that binding plus an nn.Module shell with the reference's constructor
 * signature (conformer_encoder.py:111-132) and state_dict key layout.
 *
 * Threading: a handle is bound to one CUDA device and is not thread-safe; distinct handles are independent
 * (no process-wide state).  Multi-GPU = one handle per GPU (one process or host thread each).
 */
#ifndef CFB_H_
#define CFB_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define CFB_API __attribute__((visibility("default")))
#else
#define CFB_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cfb_handle cfb_handle;
typedef void* cfb_stream; /* a cudaStream_t; NULL = the legacy default stream */

typedef enum cfb_status {
  CFB_OK = 0,
  CFB_ERR_INVALID_ARG = 1,   /* bad pointer / shape / enum value                                  */
  CFB_ERR_UNSUPPORTED = 2,   /* configuration outside the supported surface (SURVEY.md 8(a) a13)   */
  CFB_ERR_MISSING_WEIGHT = 3,/* cfb_finalize_weights: a required state_dict key was never set     */
  CFB_ERR_CUDA = 4,          /* a CUDA runtime / driver call failed                               */
  CFB_ERR_WORKSPACE = 5,     /* workspace too small or misaligned                                 */
  CFB_ERR_STATE = 6          /* call order violated (e.g. forward before finalize)                */
} cfb_status;

typedef enum cfb_dtype { CFB_F32 = 0, CFB_BF16 = 1, CFB_F16 = 2, CFB_I64 = 3, CFB_I32 = 4 } cfb_dtype;

/* Arithmetic of the forward pass. */
typedef enum cfb_precision {
  CFB_PREC_BF16 = 0,         /* product path: tcgen05 bf16 x bf16 -> fp32 tensor-core kernels, fp32 residual stream */
  CFB_PREC_FP32_VALIDATE = 1 /* validation path: the same dataflow on fp32 CUDA-core kernels (slow; tests only) */
} cfb_precision;

/* Mirrors the keyword arguments of ConformerEncoder.__init__ (conformer_encoder.py:111-132).  Dropouts are
 * identity at inference and have no field.  Unsupported values make cfb_create return CFB_ERR_UNSUPPORTED. */
typedef struct cfb_config {
  int32_t feat_in;                   /* mel bins, e.g. 80; 1 ... 359                                          */
  int32_t n_layers;
  int32_t d_model;
  int32_t feat_out;                  /* -1 (or == d_model): no out_proj (conformer_encoder.py:209-214)         */
  int32_t subsampling_factor;        /* power of two >= 2; 'striding' is the only supported scheme             */
  int32_t subsampling_conv_channels; /* -1 = d_model                                                           */
  int32_t ff_expansion_factor;
  int32_t n_heads;                   /* head dimension d_model / n_heads even and <= 128 (heads <= 64 wide are   */
                                     /* padded to 64 columns, wider ones to 128)                               */
  int32_t conv_kernel_size;          /* odd, <= 31 + ... (depth-wise taps)                                     */
  int32_t xscaling;                  /* 1: multiply pre_encode output by sqrt(d_model) (multi_head_attention.py:305) */
  int32_t precision;                 /* cfb_precision                                                          */
  int32_t reserved[5];
} cfb_config;

/* ---- lifetime ------------------------------------------------------------------------------------------------ */

/* Creates an encoder instance on CUDA device `device`.  Replaces ConformerEncoder.__init__. */
CFB_API int cfb_create(const cfb_config* cfg, int device, cfb_handle** out);
CFB_API void cfb_destroy(cfb_handle* h);
/* Text of the last error on this handle (or of the last failed cfb_create when h == NULL). Never NULL. */
CFB_API const char* cfb_last_error(const cfb_handle* h);

/* ---- weights (replaces load_state_dict; nemo/core/connectors/save_restore_connector.py:163-165) ----------------- */

/* Copies one tensor of the reference state_dict, addressed by its reference key (e.g.
 * "layers.3.self_attn.linear_q.weight"), from host or device memory.  dtype: CFB_F32 / CFB_BF16 / CFB_F16.
 * Keys ending in "num_batches_tracked" are accepted and ignored.  The extra key "pos_enc.div_term"
 * (d_model/2 floats) optionally overrides the sinusoid frequencies (multi_head_attention.py:238-241). */
CFB_API int cfb_set_weight(cfb_handle* h, const char* ref_key, const void* host_or_dev_ptr, int dtype,
                   const int64_t* shape, int ndim);
/* Validates that every required key is present and packs the device arena: BatchNorm folded into the
 * depth-wise taps, sqrt(d_model) folded into pre_encode.out, q/k/v concatenated, GLU rows interleaved,
 * conv kernels re-ordered for the implicit GEMM, bf16 copies made.  May allocate and synchronise. */
CFB_API int cfb_finalize_weights(cfb_handle* h);

/* ---- forward ----------------------------------------------------------------------------------------------------- */

/* Output time extent for an input of T frames: T' = repeated floor((T-1)/2)+1. */
CFB_API int cfb_output_frames(const cfb_handle* h, int T, int* t_out);
/* Bytes of scratch cfb_forward needs for a (B, feat_in, T) batch. */
CFB_API int cfb_workspace_bytes(const cfb_handle* h, int B, int T, size_t* out);

/* Enqueues the whole forward pass on `stream`.  No allocation, no host<->device synchronisation, CUDA-graph
 * capturable.  All pointers are device pointers.
 *   feats        (B, feat_in, T) row-major, CFB_F32 or CFB_BF16                       [audio_signal]
 *   lengths      (B,) int64 valid frame counts, or NULL = all rows are T long        [length]
 *   encoded      (B, T', d_out) row-major (the reference returns its (B, d_out, T') transposed view,
 *                conformer_encoder.py:280), CFB_F32 or CFB_BF16; frames t >= encoded_len[b] are written as 0
 *   encoded_len  (B,) int32 = calc_length(lengths) (subsampling.py:272-282), bit-exact
 *   workspace    >= cfb_workspace_bytes(B, T), 256-byte aligned
 */
CFB_API int cfb_forward(cfb_handle* h, const void* feats, int feats_dtype, const int64_t* lengths, int B, int T,
                void* encoded, int out_dtype, int32_t* encoded_len, void* workspace, size_t ws_bytes,
                cfb_stream stream);

/* Variable-length ("packed") form of cfb_forward: same inputs, same outputs, and bit-identical results on every
 * frame t < encoded_len[b] (frames behind it are zeros, as in cfb_forward) -- but no arithmetic is spent on padding.
 * Each utterance occupies its own slot of token rows (its T'_b frames + a >= 15-row gap), so LayerNorm / GEMM kernels run
 * over sum_b T'_b rows instead of B * T'max, attention works per slot, and the strided convolutions reproduce the
 * reference's padded-batch edge effect (subsampling.py:172-175 runs them over the padded batch: the frame behind a short
 * utterance is conv(zero-extended input), the one behind the longest is the convolution's zero padding).  This is what
 * a length-bucketed shard of a mixed-length batch runs (SURVEY.md 8(e); the reference pads: audio_to_text.py:48-99).
 *   lengths       (B,) int64 on the DEVICE (or NULL = all rows T long), as for cfb_forward
 *   lengths_host  the same values in HOST memory: sizes the grids and the workspace; read during the call only
 * Enqueue-only like cfb_forward (no allocation, no synchronisation, capturable: a captured graph is valid for these
 * lengths).  CFB_ERR_UNSUPPORTED for the fp32 validation precision and for encoders with out_proj. */
CFB_API int cfb_packed_workspace_bytes(const cfb_handle* h, const int64_t* lengths_host, int B, int T, size_t* out);
CFB_API int cfb_forward_packed(cfb_handle* h, const void* feats, int feats_dtype, const int64_t* lengths,
                       const int64_t* lengths_host, int B, int T, void* encoded, int out_dtype, int32_t* encoded_len,
                       void* workspace, size_t ws_bytes, cfb_stream stream);

/* Where an intermediate lives inside the workspace of a (B, T) cfb_forward (tests / debugging): name is one of
 * "y1" "y2" "x" "a" "h" "qkv" "ctx" "g" "c" "pe" "pos".  Offsets are bytes from the workspace base.  A bf16 batch of
 * B >= 8 runs as two half-batches, each with a workspace layout of its own, so for it the call returns
 * CFB_ERR_INVALID_ARG: ask for B <= 7, or use CFB_PREC_FP32_VALIDATE (never split). */
CFB_API int cfb_debug_buffer(const cfb_handle* h, int B, int T, const char* name, size_t* offset, size_t* bytes);

/* Per-kernel timing (bench.py's roofline): when on, cfb_forward brackets every launch with CUDA events on the
 * forward's own stream (still enqueue-only).  cfb_profile_report synchronises on the recorded events, writes one
 * line per kernel label "label<TAB>launches<TAB>total_ms\n" for everything recorded since the last report into
 * buf (NUL-terminated, truncated to cap) and clears the records. */
CFB_API int cfb_set_profiling(cfb_handle* h, int on);
CFB_API int cfb_profile_report(cfb_handle* h, char* buf, size_t cap);

/* Number of kernels the last cfb_forward call enqueued (for bench.py's gpu_launches). */
CFB_API int cfb_last_launch_count(const cfb_handle* h);

/* ---- kernel-level entry points (unit tests and composition; all enqueue-only on `stream`) ------------------------- */

typedef enum cfb_epilogue {
  CFB_EPI_LINEAR = 0, /* out = acc + bias                        (linear_pos, pre_encode.out, out_proj)   */
  CFB_EPI_SWISH = 1,  /* out = silu(acc + bias)                  (feed_forward.linear1; conformer_modules.py:196-197) */
  CFB_EPI_RELU = 2,   /* out = relu(acc + bias)                  (subsampling conv; subsampling.py:106-115) */
  CFB_EPI_RESID = 3,  /* resid += alpha * (acc + bias), fp32     (linear2 / linear_out / pointwise_conv2)  */
  CFB_EPI_QKV = 4,    /* [q+u | q+v | k | v] from a fused q/k/v projection (multi_head_attention.py:183-193) */
  CFB_EPI_GLU = 5     /* out = a * sigmoid(g), zeroed at padded frames (conformer_modules.py:162-166)       */
} cfb_epilogue;

/* D = A (M x K, row-major, lda) * W^T (W: N x K row-major, ldw) with the selected epilogue.
 * use_tensor_cores != 0: A/W are bf16 and the tcgen05 kernel runs; == 0: A/W are fp32 and the CUDA-core
 * validation kernel runs (raw accumulators go through `scratch`, M*N floats).
 * bias2 only for QKV.  lens/frames_per_seq (row r belongs to sequence r / frames_per_seq) zero the rows at frames
 * t >= lens[seq] for LINEAR, SWISH, RELU and GLU; RESID and QKV ignore them.
 * For QKV and GLU, N counts accumulator columns (3*Dp resp. 2*d) and `out` has 4*Dp resp. d columns.
 * Accepted combinations (anything else returns before enqueueing anything):
 *   out_dtype    CFB_F32 or CFB_BF16 (else CFB_ERR_UNSUPPORTED); RESID: CFB_F32 only, and with use_tensor_cores
 *                the other epilogues except LINEAR: CFB_BF16 only (CFB_ERR_UNSUPPORTED);
 *   QKV          qkv_dp > 0, qkv_dp % 64 == 0, N == 3 * qkv_dp (CFB_ERR_INVALID_ARG);
 *   GLU          N % 32 == 0 (CFB_ERR_INVALID_ARG);
 *   ldo          >= the output's column count: N, 4*Dp for QKV, N/2 for GLU (CFB_ERR_INVALID_ARG);
 *   epilogue     a cfb_epilogue value (CFB_ERR_INVALID_ARG). */
CFB_API int cfb_op_gemm(int use_tensor_cores, int epilogue, const void* A, int64_t lda, const void* W, int64_t ldw,
                const float* bias, const float* bias2, int M, int N, int K, void* out, int64_t ldo, int out_dtype,
                float alpha, const int32_t* lens, int frames_per_seq, int qkv_dp, float* scratch,
                cfb_stream stream);

/* y = LayerNorm(x) * gamma + beta over the last dim (eps 1e-5; conformer_modules.py:60-86). x fp32 (rows x d);
 * out_dtype CFB_BF16 / CFB_F32.  lens != NULL: rows at frames >= lens[seq] are written as zeros. */
CFB_API int cfb_op_layernorm(const float* x, const float* gamma, const float* beta, void* out, int out_dtype, int rows,
                     int d, const int32_t* lens, int frames_per_seq, cfb_stream stream);

/* norm_out of one layer followed by norm_feed_forward1 of the next (conformer_modules.py:120, :98) in one pass:
 * out1 = LayerNorm(x; g1, b1) fp32 (may alias x), out2 = LayerNorm(out1; g2, b2) bf16.  rows x d, d % 4 == 0, d <= 1024. */
CFB_API int cfb_op_layernorm_dual(const float* x, const float* g1, const float* b1, float* out1, const float* g2,
                                  const float* b2, void* out2_bf16, int rows, int d, cfb_stream stream);

/* Depth-wise time convolution with folded BatchNorm + Swish (conformer_modules.py:168-177).
 * x, out: (B, T, d) in `dtype` (CFB_BF16 / CFB_F32); taps (ksize, d) fp32, tap-major; bias (d) fp32; zero padding at
 * both ends of every sequence. */
CFB_API int cfb_op_depthwise(const void* x, const float* taps, const float* bias, void* out, int dtype, int B, int T, int d,
                     int ksize, cfb_stream stream);

/* Tail of the convolution module in one kernel (conformer_modules.py:168-180 + the residual add of :114):
 *   x[b,t,:] += W2 * swish(taps32[31] + sum_k taps32[k] * g[b, t + k - 15, :]) + bias2
 * g (B, T, d) bf16 (GLU output, padded frames zeroed); taps32 (32, d) fp32 = 31 BatchNorm-folded taps (shorter kernels
 * centred and zero padded) + the folded bias as row 31; W2 (d, d) bf16 = pointwise_conv2.weight; bias2 (d) fp32;
 * x (B, T, d) fp32, updated in place.  d must be a multiple of 64 and <= 512.  Bit-identical to cfb_op_depthwise
 * followed by cfb_op_gemm(CFB_EPI_RESID). */
CFB_API int cfb_op_dw_pw2(const void* g, const float* taps32, const void* W2, const float* bias2, float* x, int B, int T,
                  int d, cfb_stream stream);

/* Log-mel front-end: FilterbankFeatures.forward in eval mode (parts/preprocessing/features.py:358-453) for hann /
 * per_feature / log-add / power-2 recipes: pre-emphasis, centred STFT with reflect padding, |.|^2, mel projection,
 * log(x + log_guard), per-(utterance, mel) mean / unbiased-std normalisation over the valid frames, zeros after them.
 * audio (B, L) fp32 (L > n_fft / 2), lengths (B) int64 samples; window (win_length <= n_fft) fp32; n_fft must be 512;
 * fb (n_mels <= 96, n_fft / 2 + 1) = the `featurizer.fb` buffer, fb_span (n_mels, 2) int32 = first non-zero bin and
 * bin count of every filter (the kernel sums each filter over its own bins only); features (B, n_mels, T_out) fp32 with
 * T_out >= 1 + L / hop (the caller rounds up to `pad_to`); seq_len (B) int64 = floor(len / hop) + 1; *flag is set to 1
 * if some utterance has exactly one frame (the reference raises ValueError there).  All pointers are device pointers. */
CFB_API int cfb_op_logmel(const float* audio, const int64_t* lengths, int B, int L, const float* window, int win_length,
                  int n_fft, int hop, const float* fb, const int32_t* fb_span, int n_mels, float preemph, float log_guard, float std_eps,
                  float* features, int T_out, int64_t* seq_len, int32_t* flag, cfb_stream stream);

/* The same front end with normalize = "None" (what buffered inference builds: features.py normalize_batch returns x
 * unchanged): log-mel values as they are, frames t >= seq_len set to 0.  Same arguments as cfb_op_logmel without std_eps
 * and flag (no statistics, so a one-frame utterance is not an error). */
CFB_API int cfb_op_logmel_raw(const float* audio, const int64_t* lengths, int B, int L, const float* window, int win_length,
                      int n_fft, int hop, const float* fb, const int32_t* fb_span, int n_mels, float preemph, float log_guard,
                      float* features, int T_out, int64_t* seq_len, cfb_stream stream);

/* Buffered long-audio inference (streaming_utils.py:455-684, AudioFeatureIterator + FeatureFrameBufferer): the normalised
 * overlapping windows of many files in one launch, ready to be the encoder's audio_signal.
 *   features      (n_files, F, T) fp32 raw log-mel features (cfb_op_logmel_raw);  seq_len (n_files) int64 valid frames n
 *   first_window  (n_files) int32, ascending: file f owns windows first_window[f] ... first_window[f+1] - 1 (the last file
 *                 up to n_windows - 1); a file has n / frame_len + 1 windows
 *   out           (n_windows, F, buffer_len) fp32.  Column j of the file's window k is frame s = (k+1) frame_len -
 *                 buffer_len + j: -16.635 (log-mel silence) for s < 0, features[:, s] for s < n, 0 after; then each
 *                 (window, mel) row becomes (x - mean) / (std + 1e-5), mean and population std over its buffer_len columns.
 * 1 <= frame_len <= buffer_len.  Enqueue-only on `stream`; all pointers are device pointers. */
CFB_API int cfb_op_feature_buffers(const float* features, int n_files, int F, int T, const int64_t* seq_len,
                           const int32_t* first_window, int n_windows, int frame_len, int buffer_len, float* out,
                           cfb_stream stream);

/* Relative-position multi-head attention core (multi_head_attention.py:195-210 + :104-113), everything between the
 * q/k/v projections and linear_out:
 *   qkv  (B*T, 4*Dp): [q+u | q+v | k | v], head h at columns h*dkp .. h*dkp+dk-1 of each part (Dp = H*dkp)
 *   pos  (2T-1 rows, ld_pos): linear_pos(pos_emb) for this layer, same head packing, row k <-> relative position T-1-k
 *   ctx  (B*T, Dp): softmax((q+u)k^T + rel_shift((q+v)p^T)) / sqrt(dk)) v, keys >= lens[b] excluded, query rows
 *        >= lens[b] written as zeros.
 * use_tensor_cores != 0: bf16 in/out, fused flash-style tcgen05 kernel (no T x T matrix in HBM) for dkp 64 or 128 with
 *   1 <= dk <= dkp (pad columns dk..dkp-1 of q, k, v and pos must be zero), anything else returns CFB_ERR_INVALID_ARG;
 *   == 0: fp32 CUDA-core kernel (any dkp). */
CFB_API int cfb_op_rel_attention(int use_tensor_cores, const void* qkv, const void* pos, int64_t ld_pos, void* ctx,
                         const int32_t* lens, int B, int T, int H, int dk, int dkp, cfb_stream stream);

/* encoded_len = calc_length(lengths) repeated n_stages times (subsampling.py:272-282), float32 arithmetic inside. */
CFB_API int cfb_op_lengths(const int64_t* lengths, int32_t* out, int B, int T_full, int n_stages, cfb_stream stream);

/* ---- CTC head on the encoder output (the caller right after the path; SURVEY.md 8(f) rank 1) -----------------------
 * ConvASRDecoder (modules/conv_asr.py:437-444): logprobs = log_softmax(x W^T + b) over the V+1 classes, and the greedy
 * argmax the CTC models take next (models/ctc_models.py:593-594).
 *   x        (M, d) rows = frames (the contiguous (B, T', d) encoder output), CFB_F32 or CFB_BF16
 *   W        (v1, d) bf16 row-major = decoder_layers.0.weight[:, :, 0];  bias (v1) fp32
 *   logprobs (M, v1) fp32;  best (M) int32 = argmax over classes (first index on ties), may be NULL
 *   scratch  >= cfb_ctc_head_scratch_bytes(M, d, v1), 256-byte aligned.  Enqueue-only on `stream`. */
CFB_API size_t cfb_ctc_head_scratch_bytes(int M, int d, int v1);
CFB_API int cfb_op_ctc_head(const void* x, int x_dtype, const void* W, const float* bias, int M, int d, int v1,
                    float* logprobs, int32_t* best, void* scratch, size_t scratch_bytes, cfb_stream stream);
/* Greedy CTC collapse of the arg-max frames on the device (metrics/wer.py:152-164): per utterance b, the frames t < lens[b]
 * (all T when lens == NULL) whose class is not `blank` and differs from the previous frame's are kept, in order.
 *   best (B, T) int32;  tokens (B, T) int32 (the first n_tokens[b] entries of row b are valid);  n_tokens (B) int32. */
CFB_API int cfb_op_ctc_collapse(const int32_t* best, const int32_t* lens, int B, int T, int blank, int32_t* tokens,
                        int32_t* n_tokens, cfb_stream stream);

/* ---- Transducer greedy decode on the encoder output (the transducer recipes' consumer; SURVEY.md 8(f) rank 4) -------
 * RNNTDecoder.predict (modules/rnnt.py:190-283: Embedding with the blank as padding row + one LSTM layer), RNNTJoint.joint
 * (modules/rnnt.py:951-1008) and GreedyBatchedRNNTInfer._greedy_decode_blank_as_pad
 * (parts/submodules/rnnt_greedy_decoding.py:454-616) in one persistent cooperative kernel (csrc/rnnt_greedy.cu).
 * All weight pointers are DEVICE fp32 tensors in the reference state_dict layout:
 *   embed  prediction.embed.weight (V+1, H), row V (= blank) must be the zero padding row
 *   w_ih / w_hh / b_ih / b_hh  prediction.dec_rnn.lstm.{weight_ih,weight_hh,bias_ih,bias_hh}_l0  (4H, H) / (4H)
 *   w_pred (J, H), b_pred (J) = joint.pred;  w_enc (J, E), b_enc (J) = joint.enc;  w_out (V+1, J), b_out = joint.joint_net[-1]
 * activation: 0 relu, 1 sigmoid, 2 tanh (rnnt.py:1026-1037). */
typedef struct cfb_rnnt_weights {
  int32_t enc_hidden, pred_hidden, joint_hidden, num_classes_with_blank, activation, reserved[3];
  const float *embed, *w_ih, *w_hh, *b_ih, *b_hh, *w_pred, *b_pred, *w_enc, *b_enc, *w_out, *b_out;
} cfb_rnnt_weights;

CFB_API size_t cfb_rnnt_greedy_scratch_bytes(int enc_hidden, int pred_hidden, int joint_hidden, int B, int T);
/*   encoded      (B, T, E) row-major = the contiguous encoder output, CFB_F32 or CFB_BF16;  encoded_len (B) int32
 *   max_symbols  symbols per frame (decoding.greedy.max_symbols; <= 0: no limit)
 *   tokens, timesteps (B, max_tokens) int32 = Hypothesis.y_sequence / .timestep;  n_tokens (B)
 *   scores       (B) sum of the winning joint outputs (raw logits: the reference's CUDA branch, rnnt_greedy_decoding.py:181-183)
 *   h_out, c_out (B, H) = Hypothesis.dec_state (the LSTM state after the last emitted symbol; zeros if none)
 *   flags        (1) int32, caller-zeroed; bit 0 is set if some utterance produced more than max_tokens symbols
 *                (n_tokens keeps counting, the surplus is not stored); bit 1 if max_symbols <= 0 and some frame emitted
 *                4096 symbols (a runaway the reference would never return from; the frame is then advanced)
 *   scratch      >= cfb_rnnt_greedy_scratch_bytes(...), 256-byte aligned.  Enqueue-only on `stream`; needs a device
 *                that supports cooperative launches and whose SMs together hold the fp32 weights in shared memory
 *                (CFB_ERR_UNSUPPORTED otherwise). */
CFB_API int cfb_op_rnnt_greedy(const cfb_rnnt_weights* w, const void* encoded, int x_dtype, const int32_t* encoded_len, int B,
                       int T, int max_symbols, int max_tokens, int32_t* tokens, int32_t* timesteps, int32_t* n_tokens,
                       float* scores, float* h_out, float* c_out, int32_t* flags, void* scratch, size_t scratch_bytes,
                       cfb_stream stream);

/* ---- Transducer beam search on the encoder output (decoding.strategy = beam, search_type = default) ---------------------
 * BeamRNNTInfer.default_beam_search, and greedy_search for beam_size == 1, with sort_nbest, run for every utterance of the
 * batch (parts/submodules/rnnt_beam_decoding.py; restated in oracle/rnnt_beam_oracle.py) in one persistent cooperative
 * kernel (csrc/rnnt_beam.cu).  Same weights (cfb_rnnt_weights) and joint.enc GEMM as cfb_op_rnnt_greedy.
 * Capacities bound the per-utterance device state; an utterance that would exceed one stops and sets flags bit 0, and the
 * caller runs the call again with larger capacities (stats tells how much was used). */
typedef struct cfb_rnnt_beam_caps {
  int32_t max_expansions; /* hypotheses expanded per frame; also the n-best rows per utterance of the outputs        */
  int32_t max_hyps;       /* entries of each of the `hyps` / `kept` lists (<= 2048; kept in shared memory)           */
  int32_t max_nodes;      /* prefix-tree nodes per utterance (one per non-blank extension, plus the initial blank)    */
  int32_t max_states;     /* prediction-network outputs per utterance (one per distinct label sequence expanded)      */
  int32_t max_len;        /* labels per output hypothesis (y_sequence, its leading blank included)                    */
  int32_t reserved[3];
} cfb_rnnt_beam_caps;

CFB_API size_t cfb_rnnt_beam_scratch_bytes(int enc_hidden, int pred_hidden, int joint_hidden, int num_classes_with_blank, int B,
                                   int T, const cfb_rnnt_beam_caps* caps);
/*   encoded      (B, T, E) row-major = the contiguous encoder output, CFB_F32 or CFB_BF16;  encoded_len (B) int32
 *   beam_size    BeamRNNTInfer's beam_size (>= 1; 1 = greedy_search, up to 5 labels per frame);  beam = min(beam_size, V + 1)
 *                hypotheses end a frame, beam_k = min(beam, V) non-blank candidates extend each expansion (<= 64)
 *   score_norm   sort the n-best list by score / len(y_sequence) (non-zero) or by score
 *   temperature  softmax_temperature: log_softmax(joint / temperature) (> 0)
 *   caps         host pointer, read during the call only
 * Outputs (device), X = caps->max_expansions, L = caps->max_len; row (b, r) is the r-th hypothesis of sort_nbest's list:
 *   n_hyps       (B) int32 hypotheses in the list (0 for an utterance that stopped on a capacity)
 *   lengths      (B, X) int32 labels of each hypothesis;  tokens, timesteps (B, X, L) int32 = Hypothesis.y_sequence and
 *                .timestep (beam: the leading blank and its -1 included; greedy_search: neither)
 *   scores       (B, X) double = Hypothesis.score (accumulated in double, like the reference's Python floats)
 *   h_out, c_out (B, X, H) = Hypothesis.dec_state: the LSTM state the hypothesis's last label is predicted from (zeros for
 *                the initial hypothesis)
 *   stats        (B, 4) int32: expansions, prefix-tree nodes, state slots, most expansions at one frame
 *   flags        (1) int32, caller-zeroed; bit 0: some utterance exceeded a capacity, and which one: bit 1 max_expansions,
 *                bit 2 max_hyps, bit 3 max_nodes, bit 4 max_states, bit 5 max_len
 *   scratch      >= cfb_rnnt_beam_scratch_bytes(...), 256-byte aligned.  Enqueue-only on `stream`; CFB_ERR_UNSUPPORTED when
 *                the device has no cooperative launch, the fp32 weights and lists do not fit in the SMs' shared memory, or
 *                beam_k / max_hyps exceed the limits above. */
CFB_API int cfb_op_rnnt_beam(const cfb_rnnt_weights* w, const void* encoded, int x_dtype, const int32_t* encoded_len, int B,
                     int T, int beam_size, int score_norm, float temperature, const cfb_rnnt_beam_caps* caps,
                     int32_t* n_hyps, int32_t* lengths, int32_t* tokens, int32_t* timesteps, double* scores, float* h_out,
                     float* c_out, int32_t* stats, int32_t* flags, void* scratch, size_t scratch_bytes, cfb_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* CFB_H_ */
