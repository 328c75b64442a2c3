/*
 * vatss.h - C ABI of the B200-native VAT-SS separation hot path (libvatss_b200.so).
 *
 * The reference (teasgen/speech_separation) is pure Python/PyTorch and has no FFI or
 * plugin interface of its own (SURVEY.md §8b): its seam is Hydra `_target_` instantiation
 * of Python nn.Modules.  Every entry point below therefore cites the reference Python
 * interface it replaces (paths relative to the reference repo root), and
 * INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *  - All pointers except `params` tables are DEVICE pointers owned by the caller (PyTorch's
 *    caching allocator); the library never allocates or frees device memory.
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing
 *    synchronises the device.
 *  - Return value: 0 = OK, <0 = error; `vatss_last_error()` gives the message (thread-local).
 *  - Activations inside the library are TOKEN-MAJOR: one row of N features per frame.
 */
#ifndef VATSS_H_
#define VATSS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VATSS_ABI_VERSION 1

/* model kinds: which reference nn.Module the forward reproduces */
#define VATSS_KIND_DPTN_AV 0   /* src/model/dptn_wav.py:129-194  DPTNAVWavEncDec */
#define VATSS_KIND_DPTN_WAV 1  /* src/model/dptn_wav.py:64-113   DPTNWavEncDec   */
#define VATSS_KIND_DPTN_MASK 2 /* src/model/dptn.py:146-195      DPTNEncDec      */
#define VATSS_KIND_DPRNN 3     /* src/model/dprnn.py:230-276     DPRNNEncDec     */

/* execution engines for the dual-path blocks (shape specialisation, not a backend switch):
 * GENERIC = fp32 SIMT kernels for N <= 256, H <= 128, head dim <= 64 (W_hh in fp16 for H >= 108); TENSOR = tcgen05/TMEM kernels for the
 * production dimensions (N in {64,128}, H=128).  AUTO picks TENSOR when the shape allows. */
#define VATSS_ENGINE_AUTO 0
#define VATSS_ENGINE_GENERIC 1
#define VATSS_ENGINE_TENSOR 2
/* TENSOR engine with the DPTN block residual stream kept in fp16 only (faster, ~7e-4 instead of ~5.7e-4 rel-L2;
   ignored by the masking and DPRNN models, whose heads / un-normalised stream do not tolerate it) */
#define VATSS_ENGINE_TENSOR_F16RES 3

typedef struct vatss_model_desc {
  int32_t kind;        /* VATSS_KIND_*                                   */
  int32_t N;           /* num_features                                   */
  int32_t K;           /* kernel_size_enc (stride = K/2)                 */
  int32_t H;           /* hidden_dim of the LSTMs                        */
  int32_t num_blocks;  /* dual-path blocks                               */
  int32_t C;           /* chunk_size                                     */
  int32_t P;           /* step_size                                      */
  int32_t heads;       /* attention heads (ignored for DPRNN)            */
  int32_t bidir;       /* inter-chunk LSTM bidirectional (intra always)  */
  int32_t E;           /* video_emb_size (DPTN_AV only)                  */
  int32_t engine;      /* VATSS_ENGINE_*                                 */
  int32_t reserved;
} vatss_model_desc;

/* Canonical parameter table: host array of device pointers to fp32 tensors, in this order.
 * Names are the reference state_dict keys (SURVEY.md §8b).  Absent entries are NULL. */
enum {
  VATSS_P_ENCODER_W = 0,   /* encoder.weight (N,1,K)                                    */
  VATSS_P_DECODER_W,       /* decoder.weight (N,1,K)                                    */
  VATSS_P_VIS_W,           /* visual_compression.weight (N/2,E)                         */
  VATSS_P_VIS_B,           /* visual_compression.bias (N/2)                             */
  VATSS_P_GATE,            /* gate (1)                                                  */
  VATSS_P_VLN_W,           /* video_ln.weight (N)                                       */
  VATSS_P_VLN_B,           /* video_ln.bias (N)                                         */
  VATSS_P_PRELU,           /* dprnn.speakers_separation.0.weight (1)                    */
  VATSS_P_SPK_W,           /* dprnn.speakers_separation.1.weight (2N,N,1,1)             */
  VATSS_P_SPK_B,           /* dprnn.speakers_separation.1.bias (2N)                     */
  VATSS_P_HEAD_W,          /* dprnn.postprocessing.0.weight | dprnn.output.0.weight (N,N,1) */
  VATSS_P_HEAD_B,          /* ... bias (N)                                              */
  VATSS_P_HGATE_W,         /* dprnn.output_gate.0.weight (N,N,1)   (DPTN_MASK only)     */
  VATSS_P_HGATE_B,         /* dprnn.output_gate.0.bias (N)                              */
  VATSS_P_GLOBAL_COUNT
};
/* per sub-block (blocks x {intra,inter}), prefix dprnn.model.<i>.{intra,inter}_chunk_block. */
enum {
  VATSS_S_INPROJ_W = 0, /* mha.in_proj_weight (3N,N)        (NULL for DPRNN)   */
  VATSS_S_INPROJ_B,     /* mha.in_proj_bias (3N)                               */
  VATSS_S_OUTPROJ_W,    /* mha.out_proj.weight (N,N)                           */
  VATSS_S_OUTPROJ_B,    /* mha.out_proj.bias (N)                               */
  VATSS_S_LN1_W,        /* ln1.weight (N)                                      */
  VATSS_S_LN1_B,        /* ln1.bias (N)                                        */
  VATSS_S_WIH,          /* rnn.weight_ih_l0 (4H,N)                             */
  VATSS_S_WHH,          /* rnn.weight_hh_l0 (4H,H)                             */
  VATSS_S_BIH,          /* rnn.bias_ih_l0 (4H)                                 */
  VATSS_S_BHH,          /* rnn.bias_hh_l0 (4H)                                 */
  VATSS_S_WIH_R,        /* rnn.weight_ih_l0_reverse (NULL if unidirectional)   */
  VATSS_S_WHH_R,
  VATSS_S_BIH_R,
  VATSS_S_BHH_R,
  VATSS_S_FFN_W,        /* ffn.1.weight | fc.weight (N, H*(1+bidir))           */
  VATSS_S_FFN_B,        /* ffn.1.bias | fc.bias (N)                            */
  VATSS_S_LN2_W,        /* ln2.weight | norm1d.weight (N)                      */
  VATSS_S_LN2_B,        /* ln2.bias | norm1d.bias (N)                          */
  VATSS_S_COUNT
};
/* table length = VATSS_P_GLOBAL_COUNT + num_blocks*2*VATSS_S_COUNT;
 * entry(block b, path p in {0 intra,1 inter}, slot s) = GLOBAL_COUNT + (2*b+p)*S_COUNT + s */

const char* vatss_last_error(void);
int vatss_abi_version(void);
/* NULL when the model runs on the tcgen05 TENSOR engine (or engine = GENERIC was requested); otherwise the reason why
 * engine = AUTO / TENSOR falls back to the fp32 SIMT engine (a ~20x slower path: the Python face warns once).
 * No reference counterpart: the reference has one execution path (src/model/dptn_wav.py:171-194). */
const char* vatss_engine_fallback_reason(const vatss_model_desc* d);

/* Geometry helpers (exact integer index maths of the reference).
 *   L = (T-K)/(K/2)+1      nn.Conv1d output length        src/model/dptn_wav.py:153
 *   S = (L-C)/P+1          F.unfold, no padding           src/model/dprnn.py:131-135 */
int vatss_frames(const vatss_model_desc* d, int T);
int vatss_chunks(const vatss_model_desc* d, int L);

/* Bytes of caller-provided scratch needed by vatss_forward for this shape. */
size_t vatss_workspace_bytes(const vatss_model_desc* d, int B, int T, int Tv);
/* Bytes of the packed-weight buffer used by the TENSOR engine (0 if GENERIC only). */
size_t vatss_packed_weight_bytes(const vatss_model_desc* d);
/* Re-lay the fp32 parameters into the TENSOR engine's operand formats (fp16, K-major,
 * fused LSTM bias, ...).  Call once per weight update.  Replaces nothing in the reference;
 * it is the analogue of nn.LSTM.flatten_parameters() (src/model/dptn.py:44). */
int vatss_pack_weights(const vatss_model_desc* d, const float* const* params, int n_params,
                       void* packed, size_t packed_bytes, void* stream);

/* Whole forward pass.  Replaces
 *   DPTNAVWavEncDec.forward(mix, s1_embedding, s2_embedding)   src/model/dptn_wav.py:171-194
 *   DPTNWavEncDec.forward(mix)                                 src/model/dptn_wav.py:101-113
 *   DPTNEncDec.forward(mix)                                    src/model/dptn.py:183-195
 *   DPRNNEncDec.forward(mix)                                   src/model/dprnn.py:263-276
 * mix (B,T) f32; emb1/emb2 (B,E,Tv) f32 or NULL; s1_pred/s2_pred (B,T) f32 outputs. */
int vatss_forward(const vatss_model_desc* d, const float* const* params, int n_params,
                  const void* packed, const float* mix, const float* emb1, const float* emb2,
                  int B, int T, int Tv, float* s1_pred, float* s2_pred,
                  void* workspace, size_t workspace_bytes, void* stream);

/* SplitToFolds.forward  src/model/dprnn.py:122-136 : x (B,N,L) -> out (B,N,S,C), bit-exact copy */
int vatss_segment(const float* x, int B, int N, int L, int C, int P, float* out, void* stream);
/* OverlapAdd.forward    src/model/dprnn.py:145-163 : y (B,N,S,C) -> out (B,N,(S-1)P+C), plain sum */
int vatss_overlap_add(const float* y, int B, int N, int S, int C, int P, float* out, void* stream);

/* Encoder + (optional) AV fusion + token-major segmentation.
 * nn.Conv1d encoder and the gated fusion, src/model/dptn_wav.py:173-184.
 * enc_out (B,L,N) token-major; seg_out (B,S,C,N) token-major or NULL.
 * emb1/emb2 NULL -> audio only.  vis_scratch: B*Tv*N floats (AV only). */
int vatss_encoder(const vatss_model_desc* d, const float* const* params, const float* mix,
                  const float* emb1, const float* emb2, int B, int T, int Tv,
                  float* enc_out, float* seg_out, float* vis_scratch, void* stream);
/* ConvTranspose1d decoder + centred pad, src/model/dptn_wav.py:187-193.
 * u (B,L,N) token-major -> wav (B,T); proj_scratch: B*L*K floats. */
int vatss_decoder(const vatss_model_desc* d, const float* dec_w, const float* u, int B, int T,
                  float* wav, float* proj_scratch, void* stream);

/* PIT SI-SNR loss and SI-SNR / SI-SNRi metrics in one pass.
 * Replaces SiSNRLoss/BaseSSLoss.forward (src/loss/ss_losses.py:10-26,100-114) and
 * SS2BaseMetric.forward / SISNRiMetric.__call__ (src/metrics/base_metric.py:41-60,
 * src/metrics/si_snri.py:12-30).
 * Inputs (B,T) f32, mix may be NULL.  rows_out (B,6) f64: per-utterance SI-SNR in dB of the
 * pairs [s1p.s1, s2p.s2, s1p.s2, s2p.s1, mix.s1, mix.s2] (torchmetrics form, eps = FLT_EPSILON);
 * rows_loss_out (B,4) f64: per-utterance -20log10 power ratios of the first four pairs
 * (no eps, reference loss form); summary_out (8) f64:
 *   [0] loss (batch-level PIT)  [1] loss perm1  [2] loss perm2
 *   [3] SI-SNR (batch-level PIT max)  [4] SI-SNRi  [5] mean SI-SNR(mix,s1)  [6] mean SI-SNR(mix,s2)
 *   [7] B
 * scratch: B*chunks*16 doubles with chunks = vatss_sisnr_chunks(T). */
int vatss_sisnr_chunks(int T);
int vatss_pit_sisnr(const float* s1p, const float* s2p, const float* s1, const float* s2,
                    const float* mix, int B, int T, double* rows_out, double* rows_loss_out,
                    double* summary_out, double* scratch, void* stream);

/* PIT SI-SDR: torchmetrics' ScaleInvariantSignalDistortionRatio (which src/metrics/si_sdr.py wraps, zero_mean=False by
 * default) with the batch-level PIT of SS2BaseMetric.forward src/metrics/base_metric.py:53-60.  Same inputs, row order
 * and scratch (B*chunks*16 doubles) as vatss_pit_sisnr; one pass over the waveforms.  Per pair, in fp64 from the raw
 * moments: alpha = (<p,t> + eps) / (||t||^2 + eps), 10 log10((||alpha t||^2 + eps) / (||alpha t - p||^2 + eps)),
 * eps = FLT_EPSILON; zero_mean = 1 removes the means first.  rows_out (B,6) f64 (rows 4, 5 NaN when mix is NULL);
 * summary_out (7) f64: [mean (r0+r1)/2, mean (r2+r3)/2, max of the two, SI-SDRi = max - mean (r4+r5)/2, mean r4,
 * mean r5, B] (3..5 NaN when mix is NULL).  fp64 restatement: oracle/sdr_oracle.py. */
int vatss_pit_sisdr(const float* s1p, const float* s2p, const float* s1, const float* s2, const float* mix, int B,
                    int T, int zero_mean, double* rows_out, double* summary_out, double* scratch, void* stream);

/* PIT SDR / SDRi: BSS-eval SDR with a distortion filter of filter_length taps (torchmetrics' SignalDistortionRatio on
 * its direct-solve path) for the six pairings of vatss_pit_sisnr, and the summary of vatss_pit_sisdr.  Per pair, in
 * fp64: optional mean removal, both signals normalised by max(||x||, 1e-6), r[l] = sum t[n] t[n+l] and
 * b[l] = sum t[n] p[n+l] for l < filter_length (direct lag sums), r[0] += load_diag (load_diag < 0: none), the
 * symmetric Toeplitz system R x = b solved by the Levinson recursion, coh = b.x, 10 log10(coh / (1 - coh)).  A target
 * whose recursion meets a prediction error <= 0 (all zeros, or a singular R without load_diag) gets NaN rows.
 * Workspace bytes for B utterances of T samples; 0 on bad arguments (B or T <= 0, B > 65535, filter_length < 1 or
 * above 2048, T < filter_length), see vatss_last_error.  No host synchronisation; bitwise reproducible, and an
 * utterance gets the same rows alone as inside a batch.  fp64 restatement: oracle/sdr_oracle.py. */
size_t vatss_sdr_workspace_bytes(int B, int T, int filter_length);
int vatss_sdr(const float* s1p, const float* s2p, const float* s1, const float* s2, const float* mix, int B, int T,
              int filter_length, int zero_mean, double load_diag, double* rows_out, double* summary_out,
              void* workspace, size_t workspace_bytes, void* stream);

/* Gradient of summary_out[0] (the batch-level PIT loss) with respect to the two predictions: the first piece of the
 * reference's training step (`batch["loss"].backward()`, src/trainer/trainer.py:46, through BaseSSLoss.forward
 * src/loss/ss_losses.py:10-26 and SiSNRLoss.forward :100-114).  `scratch` and `summary` are those a preceding
 * vatss_pit_sisnr call on the same tensors wrote; grad_out: device pointer to the upstream scalar gradient (NULL = 1).
 * grad_s1p / grad_s2p (B,T) f32.  Targets get no gradient (they are data). */
int vatss_pit_sisnr_backward(const float* s1p, const float* s2p, const float* s1, const float* s2, int B, int T,
                             const double* scratch, const double* summary, const float* grad_out, float* grad_s1p,
                             float* grad_s2p, void* stream);

/* Stand-alone entry points of the TENSOR-engine kernels (unit tests, ncu attribution).
 * vatss_tc_gemm: out = A[M,K] (fp16, row pitch lda) x W[NOUT,K]^T (fp16) + bias with epilogue
 *   epi 0: out16 fp16 | 1: out32 (+res) | 2: out32 = LN(.+res), out16 = act16(out32) | 3: out32 = LN(.)+res
 *   (the per-token projections of src/model/dptn.py:46-51 on tcgen05 tensor cores). */
int vatss_tc_gemm(int epi, const void* A16, long long lda, const void* W16, const float* bias, const float* res,
                  long long ldr, const float* ln_w, const float* ln_b, float* out32, long long ldo32, void* out16,
                  long long ldo16, int act16, const float* prelu_a, long long M, int NOUT, int K, void* stream);

/* vatss_tc_gemm_ln16: the LayerNorm epilogue (epi 2) with the residual given as fp16 (res16, row pitch ldr16) and
 * an optional fp32 output (out32 may be NULL): out = LN(A W^T + bias + res16), out16 = act16(out) - the form the
 * DPTN sub-blocks use for `ln2(ffn(r) + a)` and, with engine TENSOR_F16RES, `ln1(mha(x) + x)` (src/model/dptn.py:47,51). */
int vatss_tc_gemm_ln16(const void* A16, long long lda, const void* W16, const float* bias, const void* res16,
                       long long ldr16, const float* ln_w, const float* ln_b, float* out32, long long ldo32,
                       void* out16, long long ldo16, int act16, const float* prelu_a, long long M, int NOUT, int K,
                       void* stream);

/* vatss_tc_lstm: nn.LSTM(N->128) recurrence (src/model/dptn.py:23-29,49) on a CTA pair, input and recurrent
 * contractions fused per time step.  x16 (B,S,C,N) fp16 token-major; params: fp32 nn.LSTM tensors of the
 * forward (and reverse, if ndir=2) direction; out16 (B*S*C, ndir*128) fp16, relu(h) if act=1.
 * mode 0 = intra-chunk sequences, 1 = inter-chunk.  wpack: ndir*512*(N+128) halfs (ndir*512*(2N+128) with x16lo),
 * bias_pack: ndir*512 floats. */
int vatss_tc_lstm(const void* x16, const void* x16lo /* NULL, or half(x - half(x)): hi/lo split variant, N = 64 */,
                  const float* const* lstm_params /* [8]: Wih,Whh,bih,bhh fwd then rev */,
                  void* out16, int mode, int B, int S, int C, int N, int ndir, int act, void* wpack,
                  float* bias_pack, void* stream);

/* vatss_tc_attention: softmax(q k^T) v per (sequence, head) on packed fp16 qkv (B*S*C, 3N) whose q part is
 * pre-scaled by log2(e)/sqrt(hd); out16 (B*S*C, N).  mode 0 intra / 1 inter; force_simt=1 runs the SIMT fallback. */
int vatss_tc_attention(const void* qkv16, void* out16, int mode, int B, int S, int C, int N, int heads, int force_simt,
                       void* stream);

/* Stand-alone entry points of the GENERIC-engine kernels (fp32 SIMT; unit tests).  All tensors fp32.
 * vatss_generic_gemm: out[m, n] (row pitch ldc) = act(A)[m, :] . W[n, :] + bias[n] + bias2[n] + R[m, n] for m < M,
 *   n < NOUT; A (M, K) row pitch lda, W (NOUT, K) dense, R row pitch ldr; bias, bias2, R may be NULL;
 *   act 0 none, 1 ReLU, 2 PReLU with slope *prelu_a (applied to A, as the speaker split does, dptn_wav.py:47-59). */
int vatss_generic_gemm(const float* A, long long lda, const float* W, const float* bias, const float* bias2,
                       const float* R, long long ldr, float* out, long long ldc, long long M, int NOUT, int K, int act,
                       const float* prelu_a, void* stream);
/* vatss_generic_layernorm: rows of N <= 256 features, dense; biased variance, eps 1e-5.
 *   mode 0: out = LN(in + res) (src/model/dptn.py:47,51); mode 1: out = LN(in) + res (src/model/dprnn.py:42-45);
 *   res may be NULL. */
int vatss_generic_layernorm(const float* in, const float* res, const float* w, const float* b, float* out,
                            long long rows, int N, int mode, void* stream);
/* vatss_generic_attention: softmax(q k^T / sqrt(hd)) v per (sequence, head), hd = N / heads <= 64, any length;
 * qkv (B*S*C, 3N) token-major, q unscaled (mha.in_proj output, src/model/dptn.py:16-21); out (B*S*C, N).
 * mode 0 intra-chunk sequences, 1 inter-chunk. */
int vatss_generic_attention(const float* qkv, float* out, int mode, int B, int S, int C, int N, int heads,
                            void* stream);
/* vatss_generic_lstm: the nn.LSTM recurrence (h0 = c0 = 0, gates i f g o) on pre (B*S*C, ndir*4H) = x W_ih^T + b_ih
 * + b_hh of every direction; W_hh (4H, H) per direction (whh_r NULL for ndir = 1); out (B*S*C, ndir*H) = h.
 * H a multiple of 4 up to 128; W_hh is used in fp32 for H <= 104 and rounded to fp16 for H >= 108. */
int vatss_generic_lstm(const float* pre, const float* whh_f, const float* whh_r, float* out, int mode, int B, int S,
                       int C, int H, int ndir, void* stream);

/* vatss_tc_tail: the TENSOR engine's separator tail on its own - speaker split, overlap-add with the centred pad,
 * post-conv (or masking) head and decoder - through the same dispatch vatss_forward runs after its last block.
 * x16 (B,S,C,N) fp16 token-major = PReLU(x) as the last block's epilogue writes it; enc (B,L,N) f32;
 * d / params / packed as for vatss_forward (d must select the TENSOR engine); s1_pred, s2_pred (B,T) f32;
 * workspace >= vatss_workspace_bytes(d, B, T, 0). */
int vatss_tc_tail(const vatss_model_desc* d, const float* const* params, int n_params, const void* packed,
                  const void* x16, const float* enc, int B, int T, float* s1_pred, float* s2_pred,
                  void* workspace, size_t workspace_bytes, void* stream);

/* Long recordings: overlapping windows separated as one batch, speaker order aligned between neighbouring windows and
 * crossfaded back together.  No reference counterpart: the reference separates whole fixed-length clips.
 * Geometry: window W samples, hop H with W/2 <= H < W, overlap O = W - H.  A recording of T samples has
 * n = vatss_longform_windows(T, W, H) windows (1 if T <= W, else 1 + ceil((T - W) / H)); window j covers
 * [jH, jH + W) and is zero at or past T.  Windows of R recordings are numbered w = r n + j. */
int vatss_longform_windows(int T, int W, int H);   /* n, or <0 on bad arguments */
/* Cut windows [first, first + count) of mix (R,T) into mix_out (count,W).  emb1/emb2 (R,E,Tv) or NULL: also cut the
 * embedding windows emb*_out (count,E,W/spf), window j taking frames [jH/spf, jH/spf + W/spf) with frames at or past
 * Tv repeating frame Tv-1 (spf = samples per video frame; W and H must be multiples of it). */
int vatss_window_cut(const float* mix, const float* emb1, const float* emb2, int R, int T, int Tv, int E, int W, int H,
                     int spf, int first, int count, float* mix_out, float* emb1_out, float* emb2_out, void* stream);
/* Bytes of scratch vatss_window_stitch needs for R recordings of n windows each (0 on bad arguments). */
size_t vatss_window_stitch_scratch_bytes(int R, int n);
/* y1, y2 (R n, W): the two speaker outputs of every window -> s1, s2 (R,T).  For each adjacent pair (r, j) the
 * overlap's fp64 sums [a1.b1, a1.b2, a2.b1, a2.b2, a1.a1, a2.a2, b1.b1, b2.b2] (a = window j from offset H, b = window
 * j+1 from offset 0) decide a swap when cos(a1,b2) + cos(a2,b1) > cos(a1,b1) + cos(a2,b2) (normalised correlation, 0
 * for a zero energy); window j then gives speaker s from its row s XOR (flags 0..j-1 XORed), so the output keeps
 * window 0's order.  In an overlap, position i in [0,O): (1 - a) y_j + a y_{j+1}, a = (i + 0.5) / O in fp32.
 * swaps_out (R, n-1) u8 and corr_out (R, n-1, 8) f64 may be NULL.  Bitwise reproducible. */
int vatss_window_stitch(const float* y1, const float* y2, int R, int T, int W, int H, float* s1, float* s2,
                        uint8_t* swaps_out, double* corr_out, void* scratch, size_t scratch_bytes, void* stream);

/* STOI / extended STOI of the four PIT pairings of a batch.  Replaces src/metrics/stoi.py (torchmetrics'
 * ShortTimeObjectiveIntelligibility -> pystoi 0.4 stoi(target, preds, fs, extended) on the host, one utterance at a
 * time) and the batch-level PIT of SS2BaseMetric.forward src/metrics/base_metric.py:53-60.  fp64 restatement:
 * oracle/stoi_oracle.py (ESTOI without pystoi's EPS-scale noise, so deterministic).
 * Workspace bytes for B utterances of T samples at fs Hz; 0 on bad arguments (B or T <= 0, fs outside
 * 1 .. 1000000, or a signal shorter than one 256-sample frame after resampling to 10 kHz), see vatss_last_error. */
size_t vatss_stoi_workspace_bytes(int B, int T, int fs);
/* s1p, s2p, s1, s2 (B,T) f32 at fs Hz -> rows_out (B,4) f64: [s1p.s1, s2p.s2, s1p.s2, s2p.s1] (target second);
 * kept_out (B,2) int32 or NULL: frames kept by the silent-frame removal of s1 and s2; summary_out (3,) f64:
 * [batch mean of (row0 + row1)/2, batch mean of (row2 + row3)/2, max of the two].  extended = 1 gives ESTOI.
 * No host synchronisation; bitwise reproducible and independent of the other utterances of the batch. */
int vatss_stoi(const float* s1p, const float* s2p, const float* s1, const float* s2, int B, int T, int fs, int extended,
               double* rows_out, int* kept_out, double* summary_out, void* workspace, size_t workspace_bytes,
               void* stream);

/* Instrumentation (no reference counterpart; used by bench.py).
 * vatss_launch_count: number of kernels this library has launched in this process.
 * vatss_profile_begin: start recording CUDA-event pairs around the stages of subsequent calls
 * (on the stream they are launched on); vatss_profile_end synchronises those events and returns
 * accumulated milliseconds and launch counts per stage (VATSS_STAGE_* order), then disables. */
#define VATSS_STAGE_COUNT 9
/* 0 frontend 1 qkv 2 attention 3 outproj+ln1 4 lstm-input 5 lstm-recurrent 6 ffn+ln2 7 tail 8 sisnr */
unsigned long long vatss_launch_count(void);
/* debug: device buffer (>= 128 int64) receiving a clock64 trace of CTA 0 of vatss_tc_lstm; NULL disables */
void vatss_debug_lstm_trace(void* dev_buffer);
/* debug / experiments: cap the grid of the persistent GEMM and attention kernels (0 = one CTA per SM) */
void vatss_debug_cta_limit(int ctas);
/* select the LSTM kernel of the plain fp16 path: 1 = two interleaved half tiles per CTA (default), 0 = one tile */
void vatss_debug_lstm_pingpong(int on);
/* row groups (32 sequences) per CTA of the half-tile LSTM kernel: 0 = automatic (fewest waves x gate time), 2 / 3 = a
 * group occupies both 32-row slots of a half tile so the recurrence spreads over more SMs, 4 = dense 128-row tiles */
void vatss_debug_lstm_groups(int groups);
/* fused tail of the post-conv heads: 1 = rows staged through shared memory by bulk copies (default where the chunk
 * overlap is 50 %), 0 = the gather kernel (bit-identical results; cross-check) */
void vatss_debug_tail_staged(int on);
/* 1 (default): the QKV and out-projection GEMMs walk their row tiles in reverse so that they start on the part of their
 * input that the preceding kernel wrote last (L2 reuse); 0: every kernel walks forwards.  Same results. */
void vatss_debug_gemm_l2_order(int on);
/* select the tcgen05 attention kernel: 3 = P and O kept in TMEM (tc_attn3.cu, default), 1 = round-1 kernel (tc_attention.cu) */
void vatss_debug_attention_version(int v);
int vatss_profile_begin(void);
int vatss_profile_end(float* ms_per_stage, int* launches_per_stage, int n_stages);

/* ---------------------------------------------------------------------------------------------------------------
 * Lipreader front end (SURVEY.md 8f rank 4): the video feature extractor whose (512, Tv) embeddings the DPTN-AV model
 * consumes.  Replaces, for modality="video", backbone_type="resnet", extract_feats=True:
 *   Lipreading.forward(x, lengths)        src/lipreader/lipreading/model.py:252-273  (frontend3D :180-207, trunk = ResNet-18
 *                                         src/lipreader/lipreading/models/resnet.py:31-145)
 *   the "test" preprocessing pipeline     src/lipreader/lipreading/dataloaders.py:24-29 (Normalize(0,255), CenterCrop(88,88),
 *                                         Normalize(0.421,0.165)) as an affine map + crop window folded into the first load
 *   its callers                           make_embeddings.py:58-66, profiler.py:17-22, src/utils/init_utils.py:168-207
 * Parameter table: host array of VATSS_LIP_NCONV * VATSS_LIP_PSLOTS device pointers (fp32), convolution-major:
 *   conv 0            frontend3D.0 (Conv3d 64x1x5x7x7) with frontend3D.1 (BatchNorm3d) and frontend3D.2 (PReLU slopes, or NULL)
 *   conv 1+3k, 2+3k   trunk.layer<l>.<b>.conv1 / conv2 with bn1 / bn2 and relu1 / relu2 slopes (PReLU only), k = 2(l-1)+b
 *   conv 3+3k         trunk.layer<l>.<b>.downsample.0 / .1 (all six NULL where the block has no shortcut convolution)
 *   slots per conv    weight, bn.weight, bn.bias, bn.running_mean, bn.running_var, PReLU weight
 * relu_type: 1 relu, 2 prelu, 3 swish (x * sigmoid(x), models/swish.py:10).  BatchNorm uses the running statistics
 * (eval mode - the only mode the reference runs the lipreader in: make_embeddings.py:47).
 * engine: VATSS_LIP_ENGINE_F32 = fp32 FMA-pipe implicit GEMM (exact to ~1e-6 against the fp32 reference);
 *         VATSS_LIP_ENGINE_TENSOR = trunk convolutions on tcgen05 with fp16 activations, fp32 accumulation. */
#define VATSS_LIP_NCONV 25
#define VATSS_LIP_PSLOTS 6
#define VATSS_LIP_ENGINE_F32 0
#define VATSS_LIP_ENGINE_TENSOR 1
/* experiments only (tools/lipreader_ablate.py): switch parts of the tcgen05 convolution kernel off to time the rest:
 * bit 0 no gather loads, bit 1 no epilogue math / stores, bit 2 no weight TMA, bits 3-5 no stores / activation / shortcut
 * loads, bits 6-7 relaxed arrival / no proxy fence, bit 8 two instead of three CTAs per SM for 64-channel layers
 * (valid results).  0 = production. */
void vatss_debug_lipreader(int flags);
/* select the tcgen05 convolution kernel: 1 = one tile per CTA, two CTAs per SM (default; the ablation switches and the
 * trace exist in this kernel only), 2 = persistent kernel with a separate epilogue warpgroup (bit-identical results,
 * measured slower: DESIGN.md 3.7) */
void vatss_debug_lipreader_kernel(int version);
/* debug: device buffer (>= 8192 int64) receiving globaltimer / clock64 stamps of the first 1024 CTAs of every
 * following tcgen05 convolution launch (the last launch wins); NULL disables */
void vatss_debug_lipreader_trace(void* dev_buffer);
/* debug: device pointers receiving every stage of the following lipreader forwards (NULL entries skipped; NULL / 0 disables).
 * Slot 0: front end before the max pool (F, H1, W1, 64); slot 1: pooled trunk input (F, H0, W0, 64); block k = 0..7:
 * slot 2+3k conv1 output after its activation, 3+3k shortcut output (blocks with a shortcut convolution only), 4+3k block
 * output act(conv2 + residual).  Every slot holds all F = B T frames, fp32 under the f32 engine, fp16 under the tensor
 * engine.  The table is copied at the call. */
#define VATSS_LIP_NSTAGES 26
void vatss_debug_lipreader_capture(void* const* stages, int n);
size_t vatss_lipreader_packed_bytes(void);
/* scratch for B x T frames cropped to Hc x Wc (frames are processed in chunks, so this is bounded) */
size_t vatss_lipreader_workspace_bytes(int B, int T, int Hc, int Wc);
/* fold BatchNorm into per-channel scale / shift and re-lay the convolution weights (tap-major fp32, K-major fp16) */
int vatss_lipreader_pack_weights(const float* const* params, int n_params, int relu_type, void* packed,
                                 size_t packed_bytes, void* stream);
/* video (B, T, Hin, Win) f32 -> out (B, T, 512) f32.  The network sees
 * video[:, :, y0:y0+Hc, x0:x0+Wc] * pre_scale + pre_shift (pass 0, 0, Hin, Win, 1, 0 for already preprocessed input). */
int vatss_lipreader_forward(const void* packed, size_t packed_bytes, int relu_type, const float* video, int B, int T,
                            int Hin, int Win, int y0, int x0, int Hc, int Wc, float pre_scale, float pre_shift,
                            float* out, void* workspace, size_t workspace_bytes, int engine, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VATSS_H_ */
